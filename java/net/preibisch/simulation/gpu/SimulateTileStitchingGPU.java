/*
 * Tile-stitching pair generator of the reference (S/SimulateTileStitching.java:58-258) on libmvsim, with both convolved phantoms
 * resident on the GPU.
 *
 * The constructor builds the two volumes like the reference's two pool threads (:85-117): the phantom with and without the
 * half-pixel shift (simulate, S/SimulateMultiViewDataset.java:371-392), attenuate3d, convolve and Tools.adjustImage, one thread and
 * one mvsim context each, every stage on the device.  getNextPair samples the two overlapping tiles (extractSlices of
 * Views.zeroMin( Views.interval( con, min, max ) ), :152-153,174) straight from those volumes: no tile is copied or uploaded,
 * and only the two sampled tiles cross the host link.  Seeds are drawn like the Python driver (mvsim_b200.SimulateTileStitching):
 * rnd.nextInt() for the phantom, two rnd.nextInt() per pair, and tile i is keyed by new Random( seed_i ).nextLong() on Philox
 * stream i.  close() frees the GPU volumes and the two contexts.
 */
package net.preibisch.simulation.gpu;

import java.nio.FloatBuffer;
import java.util.Random;

import net.imglib2.FinalInterval;
import net.imglib2.img.Img;
import net.imglib2.type.numeric.real.FloatType;
import net.imglib2.util.Pair;
import net.imglib2.util.ValuePair;

public class SimulateTileStitchingGPU
{
	final static int lightsheetSpacing = 3;     // S/SimulateTileStitching.java:52
	final static double attenuation = 0.01;     // :53
	final static int defaultSize = 289;         // the size simulate() renders

	final Random rnd;
	final boolean halfPixelOffset;
	final long[] dims;
	final long[] overlap = new long[ 3 ];
	final long[] ctx = new long[ 2 ];           // one context per pipeline: [0] con, [1] conHalfPixel
	final long[] con = new long[ 2 ];           // the resident convolved volumes
	final long[] tile = new long[ 2 ];          // device outputs of the two tiles, on the context of the volume each is cut from
	final long[][] tileDims = new long[ 2 ][];

	public SimulateTileStitchingGPU( final Random rnd, final boolean halfPixelOffset, final double[] overlapRatio, final Img< FloatType > psf )
	{
		this( rnd, halfPixelOffset, overlapRatio, psf, defaultSize );
	}

	/** psf is normalised in place, as convolve does (S/SimulateMultiViewDataset.java:255) */
	public SimulateTileStitchingGPU( final Random rnd, final boolean halfPixelOffset, final double[] overlapRatio, final Img< FloatType > psf, final int size )
	{
		this.rnd = rnd;
		this.halfPixelOffset = halfPixelOffset;
		this.dims = new long[] { size, size, size };
		final int seed = rnd.nextInt();        // :83, the same phantom for both
		final long[] kdims = SimulateMultiViewDatasetGPU.dims( psf );
		final FloatBuffer rawPsf = SimulateMultiViewDatasetGPU.toPinned( psf );
		final FloatBuffer normPsf = Mvsim.pinnedFloats( SimulateMultiViewDatasetGPU.numElements( kdims ) );
		try
		{
			final Throwable[] failure = new Throwable[ 2 ];
			final Thread[] threads = new Thread[ 2 ];
			for ( int i = 0; i < 2; ++i )
			{
				final int p = i;
				threads[ i ] = new Thread( () -> {
					try
					{
						pipeline( p, size, seed, kdims, rawPsf, p == 0 ? normPsf : null );
					}
					catch ( final Throwable t )
					{
						failure[ p ] = t;
					}
				} );
				threads[ i ].start();
			}
			for ( final Thread t : threads )
				join( t );
			for ( final Throwable t : failure )
				if ( t != null )
				{
					close();
					throw new RuntimeException( "SimulateTileStitchingGPU: " + t.getMessage(), t );
				}
			SimulateMultiViewDatasetGPU.copyBack( normPsf, psf );
		}
		finally
		{
			Mvsim.freePinned( rawPsf );
			Mvsim.freePinned( normPsf );
		}
		for ( int d = 0; d < 3; ++d )
			overlap[ d ] = Math.round( dims[ d ] * overlapRatio[ d ] / 2 );  // :121
		for ( int i = 0; i < 2; ++i )
		{
			final long[] min = new long[ 3 ], max = new long[ 3 ];
			final FinalInterval interval = getInterval( i );
			interval.min( min );
			interval.max( max );
			tileDims[ i ] = new long[] { max[ 0 ] - min[ 0 ] + 1, max[ 1 ] - min[ 1 ] + 1, ( max[ 2 ] - min[ 2 ] ) / lightsheetSpacing + 1 };
			final long c = ctx[ source( i ) ];
			tile[ i ] = Mvsim.volumeCreate( c, tileDims[ i ] );
			if ( tile[ i ] == 0 )
			{
				final String msg = Mvsim.lastError( c );
				close();
				throw new OutOfMemoryError( "mvsim_volume_create: " + msg );
			}
		}
	}

	/** one of the reference's two pool threads (:85-114), into con[ p ] on its own context */
	private void pipeline( final int p, final int size, final int seed, final long[] kdims, final FloatBuffer rawPsf, final FloatBuffer normPsfOut )
	{
		final long c = ctx[ p ] = Mvsim.ctxCreate( Integer.getInteger( "mvsim.device", 0 ) );
		if ( c == 0 )
			throw new RuntimeException( "mvsim_ctx_create: " + Mvsim.lastError( 0 ) + " (libmvsim has no CPU fallback)" );
		final long[] tmp = new long[ 3 ];      // phantom, attenuated phantom, PSF
		try
		{
			tmp[ 0 ] = create( c, dims );
			tmp[ 1 ] = create( c, dims );
			tmp[ 2 ] = create( c, kdims );
			con[ p ] = create( c, dims );
			check( Mvsim.devSimulatePhantom( c, size, p == 1, seed, tmp[ 0 ], null ), c );
			check( Mvsim.devAttenuate( c, tmp[ 0 ], tmp[ 1 ], attenuation, SimulateMultiViewDatasetGPU.strictReference ), c );
			check( Mvsim.volumeUpload( c, tmp[ 2 ], rawPsf ), c );
			check( Mvsim.devPsfNormalize( c, tmp[ 2 ], null ), c );
			check( Mvsim.devConvolve( c, tmp[ 1 ], tmp[ 2 ], con[ p ] ), c );
			check( Mvsim.devAdjust( c, con[ p ], SimulateMultiViewDatasetGPU.minValue, SimulateMultiViewDatasetGPU.avgIntensity, null ), c );
			if ( normPsfOut != null )
				check( Mvsim.volumeDownload( c, tmp[ 2 ], normPsfOut ), c );
			check( Mvsim.ctxSynchronize( c ), c );
		}
		finally
		{
			for ( final long v : tmp )
				if ( v != 0 )
					Mvsim.volumeFree( c, v );
		}
	}

	/** two overlapping tiles (:131-189), each sampled with its own seed from the resident volume it is cut from */
	public Pair< Img< FloatType >, Img< FloatType > > getNextPair( final float snr )
	{
		final int[] seeds = new int[] { rnd.nextInt(), rnd.nextInt() };
		for ( int i = 0; i < 2; ++i )
		{
			final long[] min = new long[ 3 ], max = new long[ 3 ];
			final FinalInterval interval = getInterval( i );
			interval.min( min );
			interval.max( max );
			final long seed = snr >= 0 ? new Random( seeds[ i ] ).nextLong() : 0;
			final int s = source( i );
			check( Mvsim.devExtractInterval( ctx[ s ], con[ s ], min, max, lightsheetSpacing, snr, seed, i, tile[ i ] ), ctx[ s ] );
		}
		return new ValuePair<>( download( 0 ), download( 1 ) );
	}

	/** (:214-233): tile 0 ends at dimension/2 + overlap; tile 1 starts at dimension(0)/2 - overlap in every dimension */
	public FinalInterval getInterval( final int tile )
	{
		final long[] min = new long[ 3 ], max = new long[ 3 ];
		for ( int d = 0; d < 3; ++d )
		{
			if ( tile == 0 )
				max[ d ] = dims[ d ] / 2 + overlap[ d ];
			else
			{
				min[ d ] = dims[ 0 ] / 2 - overlap[ d ];
				max[ d ] = dims[ d ] - 1;
			}
		}
		return new FinalInterval( min, max );
	}

	/** (:191-212) */
	public double[] getCorrectTranslation()
	{
		final long[] min = new long[ 3 ];
		getInterval( 1 ).min( min );
		final double[] t = new double[] { min[ 0 ], min[ 1 ], min[ 2 ] };
		if ( halfPixelOffset )
		{
			t[ 0 ] -= 0.5;
			t[ 1 ] -= 0.5;
		}
		t[ 2 ] /= lightsheetSpacing;
		return t;
	}

	/** frees the resident volumes and the two contexts; the object cannot sample afterwards */
	public void close()
	{
		for ( int i = 0; i < 2; ++i )
		{
			final long c = ctx[ source( i ) ];
			if ( tile[ i ] != 0 )
				Mvsim.volumeFree( c, tile[ i ] );
			tile[ i ] = 0;
		}
		for ( int p = 0; p < 2; ++p )
		{
			if ( con[ p ] != 0 )
				Mvsim.volumeFree( ctx[ p ], con[ p ] );
			con[ p ] = 0;
			if ( ctx[ p ] != 0 )
				Mvsim.ctxDestroy( ctx[ p ] );
			ctx[ p ] = 0;
		}
	}

	private int source( final int tile )
	{
		return tile == 1 && halfPixelOffset ? 1 : 0;
	}

	private Img< FloatType > download( final int i )
	{
		final long c = ctx[ source( i ) ];
		final FloatBuffer buf = Mvsim.pinnedFloats( SimulateMultiViewDatasetGPU.numElements( tileDims[ i ] ) );
		try
		{
			check( Mvsim.volumeDownload( c, tile[ i ], buf ), c );
			check( Mvsim.ctxSynchronize( c ), c );
		}
		catch ( final RuntimeException | Error e )
		{
			Mvsim.freePinned( buf );
			throw e;
		}
		return SimulateMultiViewDatasetGPU.toArrayImg( buf, tileDims[ i ] );
	}

	private static long create( final long c, final long[] d )
	{
		final long v = Mvsim.volumeCreate( c, d );
		if ( v == 0 )
			throw new OutOfMemoryError( "mvsim_volume_create: " + Mvsim.lastError( c ) );
		return v;
	}

	private static void join( final Thread t )
	{
		try
		{
			t.join();
		}
		catch ( final InterruptedException e )
		{
			Thread.currentThread().interrupt();
			throw new RuntimeException( e );
		}
	}

	static void check( final int status, final long c )
	{
		if ( status == Mvsim.OK )
			return;
		final String msg = "mvsim status " + status + ": " + Mvsim.lastError( c );
		if ( status == Mvsim.EINVAL )
			throw new IllegalArgumentException( msg );
		if ( status == Mvsim.ENOMEM )
			throw new OutOfMemoryError( msg );
		throw new RuntimeException( msg );
	}
}
