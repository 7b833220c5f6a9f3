/*
 * Drop-in for the per-view acquisition methods of net.preibisch.simulation.SimulateMultiViewDataset
 * (S = src/main/java/net/preibisch/simulation of the reference):
 *
 *     axisRotation      S/SimulateMultiViewDataset.java:80
 *     rotateAroundAxis  S/SimulateMultiViewDataset.java:104
 *     extractSlices     S/SimulateMultiViewDataset.java:181, :195
 *     poissonProcess    S/SimulateMultiViewDataset.java:233
 *     convolve          S/SimulateMultiViewDataset.java:253
 *     attenuate3d       S/SimulateMultiViewDataset.java:318
 *
 * Identical static signatures; the bodies (1) copy the RandomAccessibleInterval into a pinned off-heap float buffer
 * (ArrayImg: one bulk copy of its float[]; any other view, e.g. Views.zeroMin( Views.interval( con, min, max ) ) at
 * S/SimulateTileStitching.java:153: cursor copy in flat iteration order), (2) call the C ABI of libmvsim.so through
 * Mvsim, (3) wrap the result as an ArrayImg.  simulateView / simulateViews run the whole loop body of main() (:570-585)
 * with all intermediates resident in HBM.
 *
 * Contract notes: every stage returns a NEW Img and leaves its input alone, except convolve, which normalises the caller's
 * PSF in place like :255.  The Poisson sampler is counter based (Philox); it is keyed by ONE rnd.nextLong() drawn from the
 * caller's java.util.Random, so results stay reproducible from the caller's seed and the caller's stream advances once.
 * One mvsim context per calling thread (the reference calls this path from two pool threads, S/SimulateTileStitching.java:85-117).
 */
package net.preibisch.simulation.gpu;

import java.nio.FloatBuffer;
import java.util.ArrayList;
import java.util.List;
import java.util.Random;
import java.util.concurrent.ExecutorService;

import mpicbg.models.AffineModel3D;
import net.imglib2.Cursor;
import net.imglib2.Interval;
import net.imglib2.RandomAccessibleInterval;
import net.imglib2.img.Img;
import net.imglib2.img.array.ArrayImg;
import net.imglib2.img.array.ArrayImgs;
import net.imglib2.img.basictypeaccess.array.FloatArray;
import net.imglib2.type.numeric.real.FloatType;
import net.imglib2.view.Views;

public class SimulateMultiViewDatasetGPU
{
	/** same class-static generator as the reference (S/SimulateMultiViewDataset.java:75-76) */
	final static int seed = 464232194;
	final static Random rnd = new Random( seed );
	final static float minValue = 0.0001f;   // :77
	final static float avgIntensity = 1;     // :78

	/** 1: attenuate3d loops dimension(0) steps along y like :345 (needs X <= Y); 0: loops over Y */
	public static boolean strictReference = true;

	/* ------------------------------------------------------------------ context + pinned buffers, one set per thread */

	private static final ThreadLocal< Long > CTX = new ThreadLocal< Long >()
	{
		@Override
		protected Long initialValue()
		{
			final long ctx = Mvsim.ctxCreate( Integer.getInteger( "mvsim.device", 0 ) );
			if ( ctx == 0 )
				throw new RuntimeException( "mvsim_ctx_create: " + Mvsim.lastError( 0 ) + " (libmvsim has no CPU fallback)" );
			return ctx;
		}
	};

	static long ctx() { return CTX.get(); }

	/**
	 * Keeps the FFT spectra of repeated PSFs of the calling thread's context in up to maxBytes of GPU memory (0 = off, like the
	 * reference, which rebuilds the kernel FFT in every convolve, S/SimulateMultiViewDataset.java:257).  Results are unchanged.
	 */
	public static void setPsfCache( final long maxBytes )
	{
		check( Mvsim.psfCacheConfigure( ctx(), maxBytes ) );
	}

	/** simulateViews only: Poisson counts travel from the GPU as uint16 and are widened to the FloatType images on host threads */
	public static void setCountTransport( final boolean uint16 )
	{
		check( Mvsim.ctxSetOption( ctx(), Mvsim.OPT_COUNT_TRANSPORT, uint16 ? 1 : 0 ) );
	}

	/** releases the calling thread's context (device workspaces, stream); the next call creates a new one */
	public static void closeThreadContext()
	{
		Mvsim.ctxDestroy( CTX.get() );
		CTX.remove();
	}

	static void check( final int status )
	{
		if ( status == Mvsim.OK )
			return;
		final String msg = "mvsim status " + status + ": " + Mvsim.lastError( ctx() );
		if ( status == Mvsim.EINVAL )
			throw new IllegalArgumentException( msg );
		if ( status == Mvsim.ENOMEM )
			throw new OutOfMemoryError( msg );
		throw new RuntimeException( msg );
	}

	static long[] dims( final Interval in )
	{
		if ( in.numDimensions() != 3 )
			throw new IllegalArgumentException( "3-dimensional input expected, got " + in.numDimensions() + " dimensions" );
		return new long[] { in.dimension( 0 ), in.dimension( 1 ), in.dimension( 2 ) };
	}

	static long numElements( final long[] d ) { return d[ 0 ] * d[ 1 ] * d[ 2 ]; }

	/** the float[] behind a zero-min ArrayImg< FloatType, FloatArray >, else null */
	@SuppressWarnings( "unchecked" )
	static float[] backingArray( final Object img )
	{
		if ( img instanceof ArrayImg )
		{
			final Object access = ( ( ArrayImg< ?, ? > ) img ).update( null );
			if ( access instanceof FloatArray && ( ( ArrayImg< FloatType, ? > ) img ).firstElement() instanceof FloatType )
				return ( ( FloatArray ) access ).getCurrentStorageArray();
		}
		return null;
	}

	/**
	 * RandomAccessibleInterval -> pinned buffer in ArrayImg order (x fastest).  Fast path: bulk copy of the float[];
	 * generic path: cursor copy over Views.flatIterable (strided / offset views such as S/SimulateTileStitching.java:153).
	 */
	static FloatBuffer toPinned( final RandomAccessibleInterval< FloatType > rai )
	{
		final long n = numElements( dims( rai ) );
		final FloatBuffer buf = Mvsim.pinnedFloats( n );
		final float[] array = Views.isZeroMin( rai ) ? backingArray( rai ) : null;
		if ( array != null && array.length == n )
		{
			buf.put( array );
		}
		else
		{
			final Cursor< FloatType > c = Views.flatIterable( rai ).cursor();
			for ( long i = 0; i < n; ++i )
				buf.put( c.next().get() );
		}
		buf.rewind();
		return buf;
	}

	/** pinned buffer -> new ArrayImg of the given dims (ArrayImgs.floats over a fresh float[]); the buffer is freed */
	static Img< FloatType > toArrayImg( final FloatBuffer buf, final long[] d )
	{
		final long n = numElements( d );
		if ( n > Integer.MAX_VALUE )
			throw new IllegalArgumentException( "an ArrayImg holds at most 2^31-1 elements (S/SimulateMultiViewDataset.java:109)" );
		final float[] array = new float[ ( int ) n ];
		buf.rewind();
		buf.get( array );
		Mvsim.freePinned( buf );
		return ArrayImgs.floats( array, d );
	}

	/** pinned buffer -> the caller's own image (in-place methods): flat iteration order, the order toPinned( rai ) read it in */
	static void copyBack( final FloatBuffer buf, final RandomAccessibleInterval< FloatType > target )
	{
		final long n = numElements( dims( target ) );
		buf.rewind();
		final float[] array = Views.isZeroMin( target ) ? backingArray( target ) : null;
		if ( array != null && array.length == n )
		{
			buf.get( array );
		}
		else
		{
			final Cursor< FloatType > c = Views.flatIterable( target ).cursor();
			for ( long i = 0; i < n; ++i )
				c.next().set( buf.get() );
		}
	}

	/* ------------------------------------------------------------------ the reference's public static methods */

	/** drop-in for S/SimulateMultiViewDataset.java:80-102 (host arithmetic of libmvsim: centre (max-min)/2 in long division, float-rounded angle) */
	public static AffineModel3D axisRotation( final Interval in, final int axis, final int degrees )
	{
		final double[] m = new double[ 12 ], inv = new double[ 12 ];
		final int status = Mvsim.axisRotation( dims( in ), axis, degrees, m, inv );
		if ( status != Mvsim.OK )
			throw new IllegalArgumentException( "axisRotation: axis must be 0, 1 or 2" );
		final AffineModel3D model = new AffineModel3D();
		model.set( m[ 0 ], m[ 1 ], m[ 2 ], m[ 3 ], m[ 4 ], m[ 5 ], m[ 6 ], m[ 7 ], m[ 8 ], m[ 9 ], m[ 10 ], m[ 11 ] );
		return model;
	}

	/** drop-in for S/SimulateMultiViewDataset.java:104-135 */
	public static Img< FloatType > rotateAroundAxis( final RandomAccessibleInterval< FloatType > in, final int axis, final int degrees )
	{
		final long[] d = dims( in );
		final FloatBuffer src = toPinned( in ), dst = Mvsim.pinnedFloats( numElements( d ) );
		try
		{
			check( Mvsim.rotateAxis( ctx(), src, dst, d, axis, degrees ) );
		}
		finally
		{
			Mvsim.freePinned( src );
		}
		return toArrayImg( dst, d );
	}

	/** drop-in for S/SimulateMultiViewDataset.java:181-184: the class-static generator */
	public static Img< FloatType > extractSlices( final RandomAccessibleInterval< FloatType > randomAccessible, final int inc, final float poissonSNR )
	{
		return extractSlices( randomAccessible, inc, poissonSNR, rnd );
	}

	/** drop-in for S/SimulateMultiViewDataset.java:195-231: output dims (X, Y, (Z-1)/inc+1); poissonSNR < 0 copies without noise */
	public static Img< FloatType > extractSlices( final RandomAccessibleInterval< FloatType > randomAccessible, final int inc, final float poissonSNR, final Random rnd )
	{
		if ( inc < 1 )
			throw new IllegalArgumentException( "inc must be >= 1" );
		final long[] d = dims( randomAccessible );
		final long[] dim = new long[] { d[ 0 ], d[ 1 ], ( d[ 2 ] - 1 ) / inc + 1 };
		final long seed = poissonSNR >= 0.0 ? rnd.nextLong() : 0;
		final FloatBuffer src = toPinned( randomAccessible ), dst = Mvsim.pinnedFloats( numElements( dim ) );
		try
		{
			check( Mvsim.extractSlices( ctx(), src, d, inc, poissonSNR, seed, 0, dst ) );
		}
		finally
		{
			Mvsim.freePinned( src );
		}
		return toArrayImg( dst, dim );
	}

	/** drop-in for S/SimulateMultiViewDataset.java:233-251: returns a noisy COPY (raw counts at scale (SNR/sqrt 5)^2) */
	public static Img< FloatType > poissonProcess( final RandomAccessibleInterval< FloatType > in, final float poissonSNR, final Random rnd )
	{
		final long[] d = dims( in );
		final FloatBuffer buf = toPinned( in );
		check( Mvsim.poisson( ctx(), buf, numElements( d ), poissonSNR, rnd.nextLong(), 0 ) );
		return toArrayImg( buf, d );
	}

	/** drop-in for S/SimulateMultiViewDataset.java:253-264: normalises psf IN PLACE (:255); `service` is accepted and ignored */
	public static Img< FloatType > convolve( final Img< FloatType > img, final Img< FloatType > psf, final ExecutorService service )
	{
		final long[] d = dims( img ), kd = dims( psf );
		final FloatBuffer src = toPinned( img ), k = toPinned( psf ), dst = Mvsim.pinnedFloats( numElements( d ) );
		try
		{
			check( Mvsim.convolve( ctx(), src, d, k, kd, dst ) );
			copyBack( k, psf );
		}
		finally
		{
			Mvsim.freePinned( src );
			Mvsim.freePinned( k );
		}
		return toArrayImg( dst, d );
	}

	/** drop-in for S/SimulateMultiViewDataset.java:318-364 */
	public static Img< FloatType > attenuate3d( final RandomAccessibleInterval< FloatType > randomAccessible, final double delta )
	{
		final long[] d = dims( randomAccessible );
		final FloatBuffer src = toPinned( randomAccessible ), dst = Mvsim.pinnedFloats( numElements( d ) );
		try
		{
			check( Mvsim.attenuate( ctx(), src, dst, d, delta, strictReference ) );
		}
		finally
		{
			Mvsim.freePinned( src );
		}
		return toArrayImg( dst, d );
	}

	/* ------------------------------------------------------------------ fused entries (no reference counterpart: the loop body of main) */

	/**
	 * The loop body S/SimulateMultiViewDataset.java:570-585 in one call: rotateAroundAxis( gt, axis, degrees ), attenuate3d( .., delta ),
	 * convolve( .., psf ), Tools.adjustImage( .., minValue, avgIntensity ), extractSlices( .., inc, poissonSNR, rnd ).
	 * psf is normalised in place like :255.
	 */
	public static Img< FloatType > simulateView( final RandomAccessibleInterval< FloatType > gt, final Img< FloatType > psf, final int axis,
			final int degrees, final double delta, final int inc, final float poissonSNR, final Random rnd )
	{
		if ( inc < 1 )
			throw new IllegalArgumentException( "inc must be >= 1" );
		final long[] d = dims( gt ), kd = dims( psf );
		final long[] dim = new long[] { d[ 0 ], d[ 1 ], ( d[ 2 ] - 1 ) / inc + 1 };
		final long seed = poissonSNR >= 0.0 ? rnd.nextLong() : 0;
		final FloatBuffer src = toPinned( gt ), k = toPinned( psf ), dst = Mvsim.pinnedFloats( numElements( dim ) );
		try
		{
			check( Mvsim.simulateView( ctx(), d, kd, axis, degrees, delta, minValue, avgIntensity, inc, poissonSNR, seed, 0, strictReference, src, k, dst ) );
			copyBack( k, psf );
		}
		finally
		{
			Mvsim.freePinned( src );
			Mvsim.freePinned( k );
		}
		return toArrayImg( dst, dim );
	}

	/**
	 * The view loop of main() (:567-613) for the acquisition stages: one ground truth, one PSF and one angle per view.  The ground
	 * truth is uploaded once and the download of view v overlaps the kernels of view v+1.  All PSFs must have the same dims.
	 */
	public static List< Img< FloatType > > simulateViews( final RandomAccessibleInterval< FloatType > gt, final List< Img< FloatType > > psfs,
			final int axis, final int[] degrees, final double delta, final int inc, final float poissonSNR, final Random rnd )
	{
		final int n = degrees.length;
		if ( psfs.size() != n )
			throw new IllegalArgumentException( "one PSF per view" );
		if ( inc < 1 )
			throw new IllegalArgumentException( "inc must be >= 1" );
		final List< Img< FloatType > > result = new ArrayList< Img< FloatType > >();
		if ( n == 0 )
			return result;
		final long[] d = dims( gt ), kd = dims( psfs.get( 0 ) );
		final long[] dim = new long[] { d[ 0 ], d[ 1 ], ( d[ 2 ] - 1 ) / inc + 1 };
		final long seed = poissonSNR >= 0.0 ? rnd.nextLong() : 0;
		final FloatBuffer src = toPinned( gt );
		final FloatBuffer[] k = new FloatBuffer[ n ], dst = new FloatBuffer[ n ];
		try
		{
			for ( int v = 0; v < n; ++v )
			{
				final long[] kv = dims( psfs.get( v ) );
				if ( kv[ 0 ] != kd[ 0 ] || kv[ 1 ] != kd[ 1 ] || kv[ 2 ] != kd[ 2 ] )
					throw new IllegalArgumentException( "all PSFs of one call must have the same dimensions" );
				k[ v ] = toPinned( psfs.get( v ) );
				dst[ v ] = Mvsim.pinnedFloats( numElements( dim ) );
			}
			check( Mvsim.simulateViews( ctx(), d, kd, axis, degrees, delta, minValue, avgIntensity, inc, poissonSNR, seed, 0, strictReference, src, k, dst ) );
			for ( int v = 0; v < n; ++v )
			{
				copyBack( k[ v ], psfs.get( v ) );
				result.add( toArrayImg( dst[ v ], dim ) );
				dst[ v ] = null;
			}
		}
		finally
		{
			Mvsim.freePinned( src );
			for ( int v = 0; v < n; ++v )
			{
				if ( k[ v ] != null )
					Mvsim.freePinned( k[ v ] );
				if ( dst[ v ] != null )
					Mvsim.freePinned( dst[ v ] );
			}
		}
		return result;
	}

	/**
	 * main()'s view loop with its post-acquisition chain (:567-663) in one call: for the views `views` of a dataset with the angles
	 * `angles` (all of them; the weight normalisation needs every angle), the acquired view at angle + angleOffset, the view rotated
	 * back by -angle (makeIsotropic + rotateAroundAxis, :588-591), its PSF rotated back (:593) and its normalised weights
	 * (:576, :592, :615-646).  Returns { aligned views, aligned PSFs, aligned weights } in the order of `views`.  Seeds are drawn
	 * like main(): one rnd.nextLong() per view of the whole dataset, in view order.  psfs (one per entry of `views`, same dims)
	 * are normalised in place like :255.
	 */
	public static List< List< Img< FloatType > > > simulateDataset( final RandomAccessibleInterval< FloatType > gt, final List< Img< FloatType > > psfs,
			final int[] angles, final int angleOffset, final int[] views, final double delta, final int inc, final float poissonSNR, final float osem,
			final Random rnd )
	{
		final int nAll = angles.length, n = views.length;
		if ( psfs.size() != n )
			throw new IllegalArgumentException( "one PSF per simulated view" );
		if ( inc < 1 )
			throw new IllegalArgumentException( "inc must be >= 1" );
		final long[] d = dims( gt ), kd = dims( psfs.get( 0 ) );
		final long[] iso = new long[] { d[ 0 ], d[ 1 ], ( ( d[ 2 ] - 1 ) / inc ) * inc + 1 };
		final int[] degrees = new int[ nAll ], align = new int[ nAll ];
		final long[] seeds = new long[ nAll ];
		for ( int v = 0; v < nAll; ++v )
		{
			degrees[ v ] = angles[ v ] + angleOffset;
			align[ v ] = -angles[ v ];
			seeds[ v ] = rnd.nextLong();
		}
		final FloatBuffer src = toPinned( gt );
		final FloatBuffer[] k = new FloatBuffer[ n ], view = new FloatBuffer[ n ], kview = new FloatBuffer[ n ], w = new FloatBuffer[ n ];
		final List< Img< FloatType > > views_ = new ArrayList< Img< FloatType > >(), psfs_ = new ArrayList< Img< FloatType > >(),
				weights_ = new ArrayList< Img< FloatType > >();
		try
		{
			for ( int i = 0; i < n; ++i )
			{
				final long[] kv = dims( psfs.get( i ) );
				if ( kv[ 0 ] != kd[ 0 ] || kv[ 1 ] != kd[ 1 ] || kv[ 2 ] != kd[ 2 ] )
					throw new IllegalArgumentException( "all PSFs of one call must have the same dimensions" );
				k[ i ] = toPinned( psfs.get( i ) );
				view[ i ] = Mvsim.pinnedFloats( numElements( iso ) );
				kview[ i ] = Mvsim.pinnedFloats( numElements( kd ) );
				w[ i ] = Mvsim.pinnedFloats( numElements( d ) );
			}
			check( Mvsim.simulateDataset( ctx(), d, kd, degrees, align, delta, minValue, avgIntensity, inc, poissonSNR, seeds, strictReference,
					osem, views, src, k, null, view, kview, w, null ) );
			for ( int i = 0; i < n; ++i )
			{
				copyBack( k[ i ], psfs.get( i ) );
				views_.add( toArrayImg( view[ i ], iso ) );
				psfs_.add( toArrayImg( kview[ i ], kd ) );
				weights_.add( toArrayImg( w[ i ], d ) );
				view[ i ] = kview[ i ] = w[ i ] = null;
			}
		}
		finally
		{
			Mvsim.freePinned( src );
			for ( int i = 0; i < n; ++i )
				for ( final FloatBuffer b : new FloatBuffer[] { k[ i ], view[ i ], kview[ i ], w[ i ] } )
					if ( b != null )
						Mvsim.freePinned( b );
		}
		final List< List< Img< FloatType > > > result = new ArrayList< List< Img< FloatType > > >();
		result.add( views_ );
		result.add( psfs_ );
		result.add( weights_ );
		return result;
	}

	/* ------------------------------------------------------------------ post-acquisition chain of main() */

	/** drop-in for makeIsotropic (:144-171): linear z up-sampling by inc over the mirror-single extension */
	public static Img< FloatType > makeIsotropic( final RandomAccessibleInterval< FloatType > in, final int inc )
	{
		final long[] d = dims( in );
		final long[] dim = new long[] { d[ 0 ], d[ 1 ], ( d[ 2 ] - 1 ) * inc + 1 };
		final FloatBuffer src = toPinned( in ), dst = Mvsim.pinnedFloats( numElements( dim ) );
		try
		{
			check( Mvsim.makeIsotropic( ctx(), src, d, inc, dst ) );
		}
		finally
		{
			Mvsim.freePinned( src );
		}
		return toArrayImg( dst, dim );
	}

	/** drop-in for computeWeightImage (:280-316); `delta` is unused there as well */
	public static Img< FloatType > computeWeightImage( final RandomAccessibleInterval< FloatType > randomAccessible, final double delta )
	{
		final long[] d = dims( randomAccessible );
		final FloatBuffer dst = Mvsim.pinnedFloats( numElements( d ) );
		check( Mvsim.weightImage( ctx(), d, dst ) );
		return toArrayImg( dst, d );
	}
}
