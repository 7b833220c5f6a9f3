/*
 * Thin JNI binding of libmvsim.so (include/mvsim.h) -- the Java side of the drop-in boundary.
 *
 * One native method per C entry point of the per-view acquisition path; jni/mvsim_jni.c holds the stub of each
 * (Java_net_preibisch_simulation_gpu_Mvsim_<name>).  Every compute method returns the mvsim_status (0 = OK);
 * the facades (SimulateMultiViewDatasetGPU, ToolsGPU) turn a non-zero status into an exception carrying
 * mvsim_last_error().  All volumes are direct FloatBuffers in native byte order over PINNED host memory
 * (allocPinned), laid out like an ImgLib2 ArrayImg: x fastest, idx = x + X*(y + Y*z); dims = {X, Y, Z}.
 *
 * Java 11 (the reference's CI target, .github/workflows/build-main.yml:19).  tests/test_java_boundary.py checks that every
 * native method below has a stub in jni/mvsim_jni.c and that every stub calls exported mvsim_* symbols with the arity
 * of include/mvsim.h (there is no JDK in the build image, so these files are compiled against a stand-in jni.h there).
 */
package net.preibisch.simulation.gpu;

import java.nio.Buffer;
import java.nio.ByteBuffer;
import java.nio.ByteOrder;
import java.nio.FloatBuffer;

final class Mvsim
{
	static
	{
		System.loadLibrary( "mvsim_jni" ); // links against libmvsim.so
	}

	private Mvsim() {}

	/* status codes of include/mvsim.h */
	static final int OK = 0, EINVAL = 1, ENOMEM = 2, ECUDA = 3, ENCCL = 4, EUNSUPPORTED = 5;

	/* ---- library / context ---- */
	static native int version();                                    // mvsim_version
	static native int deviceCount();                                // mvsim_device_count; -1 on failure
	static native long ctxCreate( int device );                     // mvsim_ctx_create; 0 on failure (see lastError( 0 ))
	static native void ctxDestroy( long ctx );                      // mvsim_ctx_destroy
	static native int ctxSynchronize( long ctx );                   // mvsim_ctx_synchronize
	static native String lastError( long ctx );                     // mvsim_last_error; ctx may be 0 (last error of this thread)
	static native ByteBuffer allocPinned( long bytes );             // NewDirectByteBuffer over mvsim_alloc_pinned; null on failure
	static native void freePinned( Buffer buffer );                 // mvsim_free_pinned; any view of an allocPinned buffer that starts at its base
	static native int convPaddedDims( long[] dims, long[] kdims, long[] nfftOut ); // mvsim_conv_padded_dims
	/** mvsim_ctx_set_option: OPT_COUNT_TRANSPORT (1: Poisson counts cross the host link as uint16), OPT_HOST_THREADS,
	 * OPT_Z_KERNEL (fused z kernel: 0 auto, 1 decimated inverse, 2 full spectral, 3 polyphase: A/B runs) */
	static native int ctxSetOption( long ctx, int option, long value );
	static final int OPT_COUNT_TRANSPORT = 1, OPT_HOST_THREADS = 2, OPT_Z_KERNEL = 3;
	/** mvsim_psf_cache_configure: keep the spectra of repeated PSFs in up to maxBytes of HBM (0 = off, the reference's behaviour) */
	static native int psfCacheConfigure( long ctx, long maxBytes );
	/** mvsim_psf_cache_stats: { hits, misses, entries, bytes held } */
	static native int psfCacheStats( long ctx, long[] stats4 );

	/* ---- stage entry points: one per public static method of the reference ---- */
	/** SimulateMultiViewDataset.axisRotation (S/SimulateMultiViewDataset.java:80) + createInverse() (:107); 3x4 row-major */
	static native int axisRotation( long[] dims, int axis, int degrees, double[] fwd12, double[] inv12 );
	/** rotateAroundAxis (:104) */
	static native int rotateAxis( long ctx, FloatBuffer in, FloatBuffer out, long[] dims, int axis, int degrees );
	/** attenuate3d (:318) */
	static native int attenuate( long ctx, FloatBuffer in, FloatBuffer out, long[] dims, double delta, boolean strictReference );
	/** Tools.normImage (S/Tools.java:112): in place; sumOut[0] receives the sum that was divided out */
	static native int psfNormalize( long ctx, FloatBuffer psf, long[] kdims, double[] sumOut );
	/** convolve (:253): psf is normalised IN PLACE like :255 */
	static native int convolve( long ctx, FloatBuffer img, long[] dims, FloatBuffer psf, long[] kdims, FloatBuffer out );
	/** Tools.adjustImage (S/Tools.java:143): in place; correctionOut[0] receives the factor */
	static native int adjust( long ctx, FloatBuffer img, long[] dims, float minValue, float targetAverage, double[] correctionOut );
	/** extractSlices (:195): out holds X*Y*((Z-1)/inc+1) floats */
	static native int extractSlices( long ctx, FloatBuffer in, long[] dims, int inc, float poissonSNR, long seed, long stream, FloatBuffer out );
	/** Tools.poissonProcess (S/Tools.java:73): in place on n floats */
	static native int poisson( long ctx, FloatBuffer inout, long n, double snr, long seed, long stream );
	/** loop body of main() (:570-585) with the intermediates resident on the device; psf normalised in place */
	static native int simulateView( long ctx, long[] dims, long[] kdims, int axis, int degrees, double delta, float minValue,
			float targetAverage, int inc, float poissonSNR, long seed, long stream, boolean strictReference,
			FloatBuffer gt, FloatBuffer psf, FloatBuffer out );
	/** view loop of main() (:567-613): ground truth uploaded once, the download of view v overlaps the kernels of view v+1 */
	static native int simulateViews( long ctx, long[] dims, long[] kdims, int axis, int[] degrees, double delta, float minValue,
			float targetAverage, int inc, float poissonSNR, long seed, long firstStream, boolean strictReference,
			FloatBuffer gt, FloatBuffer[] psfs, FloatBuffer[] outs );

	/**
	 * main()'s view loop with its post-acquisition chain (:567-663) for the views `views` of a dataset of degrees.length views:
	 * degrees (acquisition, angle + angleOffset), alignDegrees (rotate-back, -angle) and seeds (noise of view v, stream v) cover ALL
	 * views, since the weight normalisation needs every angle.  psfs[i], acq[i], aligned[i], alignedPsf[i] and weights[i] belong to
	 * views[i]; psfs are normalised in place; any output array, any of its elements and sumWeights may be null (not produced).
	 */
	static native int simulateDataset( long ctx, long[] dims, long[] kdims, int[] degrees, int[] alignDegrees, double delta, float minValue,
			float targetAverage, int inc, float poissonSNR, long[] seeds, boolean strictReference, float osem, int[] views,
			FloatBuffer gt, FloatBuffer[] psfs, FloatBuffer[] acq, FloatBuffer[] aligned, FloatBuffer[] alignedPsf, FloatBuffer[] weights,
			FloatBuffer sumWeights );

	/* ---- post-acquisition chain of main() ---- */
	/** makeIsotropic (:144): out holds X*Y*((Z-1)*inc+1) floats */
	static native int makeIsotropic( long ctx, FloatBuffer in, long[] dims, int inc, FloatBuffer out );
	/** computeWeightImage (:280) */
	static native int weightImage( long ctx, long[] dims, FloatBuffer out );
	/** weight normalisation of main() (:615-661), in place; sumOut may be null */
	static native int normalizeWeights( long ctx, FloatBuffer[] weights, long[] dims, float osem, FloatBuffer sumOut );

	/* ---- device-resident volumes (mvsim_volume handles cross as long; 0 = none) ----
	 * Keep intermediates in GPU memory between calls, e.g. the two convolved volumes of the tile-stitching pair generator
	 * (SimulateTileStitchingGPU): only what the caller downloads crosses the host link.  A handle belongs to the context it was
	 * created on.  Uploads and downloads are asynchronous on the context's stream for pinned buffers: ctxSynchronize before the
	 * host touches them. */
	/** mvsim_volume_create: the handle, or 0 on failure (see lastError( ctx )) */
	static native long volumeCreate( long ctx, long[] dims );
	/** mvsim_volume_free */
	static native int volumeFree( long ctx, long vol );
	/** mvsim_volume_upload: host holds at least X*Y*Z floats of the volume's dims */
	static native int volumeUpload( long ctx, long vol, FloatBuffer host );
	/** mvsim_volume_download: host holds at least X*Y*Z floats of the volume's dims */
	static native int volumeDownload( long ctx, long vol, FloatBuffer host );
	/** simulate( halfPixelOffset, rnd ) (S/SimulateMultiViewDataset.java:371-392) into a size^3 volume; nSmallOut may be null */
	static native int devSimulatePhantom( long ctx, int size, boolean halfPixelOffset, long seed, long out, long[] nSmallOut );
	/** Tools.normImage (S/Tools.java:112) in place; sumOut may be null (then the call does not synchronise) */
	static native int devPsfNormalize( long ctx, long psf, double[] sumOut );
	/** attenuate3d (:318) */
	static native int devAttenuate( long ctx, long in, long out, double delta, boolean strictReference );
	/** convolve (:253) with a PSF already normalised by devPsfNormalize */
	static native int devConvolve( long ctx, long img, long psf, long out );
	/** Tools.adjustImage (S/Tools.java:143) in place; correctionOut may be null (then the call does not synchronise) */
	static native int devAdjust( long ctx, long img, float minValue, float targetAverage, double[] correctionOut );
	/** extractSlices (:195) of Views.zeroMin( Views.interval( in, min, max ) ) (S/SimulateTileStitching.java:152-153,174) read in
	 * place: min / max inclusive (x, y, z); out dims (max0-min0+1, max1-min1+1, (max2-min2)/inc+1) */
	static native int devExtractInterval( long ctx, long in, long[] min, long[] max, int inc, float poissonSNR, long seed, long stream, long out );

	/** pinned off-heap float buffer of n elements, native byte order */
	static FloatBuffer pinnedFloats( final long n )
	{
		final ByteBuffer b = allocPinned( 4 * Math.max( n, 1 ) );
		if ( b == null )
			throw new OutOfMemoryError( "mvsim_alloc_pinned(" + 4 * n + " bytes): " + lastError( 0 ) );
		return b.order( ByteOrder.nativeOrder() ).asFloatBuffer();
	}
}
