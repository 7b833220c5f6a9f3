// CUDA backend of the FFT convolution (host logic in fft/conv_driver.h, kernels in fft/line_fft.cuh).
// Replaces convolve() S/SimulateMultiViewDataset.java:253-264 (FFTConvolution on an ExecutorService).
#include <cuda.h>
#include <stdlib.h>

#include <string.h>

#include <array>
#include <vector>

#include "ctx.h"
#include "fft/conv_driver.h"
#include "fft/fft_launch.h"

namespace mvsim {

namespace {

// cuTensorMapEncodeTiled through the runtime's driver entry point lookup (libmvsim.so does not link libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult st;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &st) != cudaSuccess || st != cudaDriverEntryPointSuccess) p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// tensor map over the PSF spectrum h = [tiles][Nz][Ny][T] complex64 seen as float32 [tiles][Nz][Ny][2T]; box = 128 kz rows of one (tile, ky)
static bool make_h_tensor_map(const float2* base, int lanes, int tiles, int nz, int ny, unsigned long long out[16])
{
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc || getenv("MVSIM_NO_TMA")) return false;
    static_assert(sizeof(CUtensorMap) == 16 * sizeof(unsigned long long), "CUtensorMap size");
    CUtensorMap m;
    const cuuint64_t dims[4] = { (cuuint64_t)(2 * lanes), (cuuint64_t)ny, (cuuint64_t)nz, (cuuint64_t)tiles };
    const cuuint64_t strides[3] = { (cuuint64_t)lanes * 8, (cuuint64_t)ny * lanes * 8, (cuuint64_t)nz * ny * lanes * 8 };
    const cuuint32_t box[4] = { (cuuint32_t)(2 * lanes), 1, (cuuint32_t)kTmaBoxRows, 1 };
    const cuuint32_t estr[4] = { 1, 1, 1, 1 };
    const CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float2*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return false;
    memcpy(out, &m, sizeof(m));
    return true;
}

// tensor map over a row-major spectrum [outer][rows][kxc] complex64 seen as float32 [outer][rows][2*kxc]; box = 256 rows of one kx tile
static bool make_rows_tensor_map(const float2* base, int lanes, int kxc, int rows, int outer, unsigned long long out[16])
{
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc || getenv("MVSIM_NO_TMA") || (kxc * 8) % 16 != 0) return false;
    CUtensorMap m;
    const cuuint64_t dims[3] = { (cuuint64_t)(2 * kxc), (cuuint64_t)rows, (cuuint64_t)outer };
    const cuuint64_t strides[2] = { (cuuint64_t)kxc * 8, (cuuint64_t)rows * kxc * 8 };
    const cuuint32_t box[3] = { (cuuint32_t)(2 * lanes), (cuuint32_t)kPrefetchBoxRows, 1 };
    const cuuint32_t estr[3] = { 1, 1, 1 };
    const CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float2*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return false;
    memcpy(out, &m, sizeof(m));
    return true;
}

static int env_int(const char* name, int dflt)
{
    const char* v = getenv(name);
    return v ? atoi(v) : dflt;
}

// L2 prefetch distance of the passes, in CTAs of launch order: a quarter of the CTAs resident on the device, i.e.
// the target CTA starts ~2 us after the prefetch was issued.  Measured on B200, config 3 (profiles/r01_notes.md): y forward
// 1.04 ms without, 0.83 at 74-100, 0.90 at 18 or 222, 1.13 at 592 (prefetched lines are evicted by the pass's own stores
// before they are used); x forward 1.09 -> 0.95 for 28..222; fused z 2.61 -> 2.49 for 36..592.  MVSIM_L2_PREFETCH=0
// switches all of them off (A/B runs).
static int prefetch_dist(int ctas_per_sm)
{
    static const int sms = [] {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n = 148;
        return n;
    }();
    static const bool on = env_int("MVSIM_L2_PREFETCH", 1) != 0;
    const int d = ctas_per_sm * sms / 4;
    return on ? (d > 1 ? d : 1) : 0;
}

static bool otf_default()
{
    static const bool on = getenv("MVSIM_H_MATERIALIZE") == nullptr;   // default: PSF spectrum computed inside the fused z pass
    return on;
}

// D' table of the decimated fused z pass (zfused_dec_table, fft/conv_driver.h), built once per (n, crop0, n_src, inc) and kept in the
// context like the twiddle tables (synchronous upload from pageable memory: the host vector may die right after)
static int get_dec_table(mvsim_ctx* ctx, int n, int crop0, int n_src, int inc, const float2** out)
{
    const std::array<int, 4> key = { n, crop0, n_src, inc };
    auto it = ctx->dec_tables.find(key);
    if (it != ctx->dec_tables.end()) { *out = it->second; return MVSIM_OK; }
    std::vector<float2> h((size_t)n);
    zfused_dec_table(n, crop0, n_src, inc, h.data());
    float2* d = nullptr;
    MVSIM_CUDA(ctx, cudaMalloc((void**)&d, sizeof(float2) * (size_t)n));
    const cudaError_t e = cudaMemcpy(d, h.data(), sizeof(float2) * (size_t)n, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(d); return cuda_fail(ctx, e, "decimation table upload"); }
    ctx->dec_tables[key] = d;
    *out = d;
    return MVSIM_OK;
}

// does MVSIM_OPT_Z_KERNEL = 0 (auto) pick the polyphase kernel where it applies?  Measured on B200 at config 3 (profiles/r02_notes.md)
constexpr bool kPolyphaseDefault = true;

struct CudaLauncher {
    mvsim_ctx* ctx;
    bool psf_phase;
    int lanes;
    bool h_on_the_fly = otf_default();

    static int x_blocks(const FftSize& s, int n_rows, bool inverse)
    {
        const int r = x_rows_per_block(s.a, s.b, inverse);
        return (n_rows + r - 1) / r;
    }
    int finish(int r, const char* what)
    {
        ctx->launches++;
        if (r == -1) return set_error(ctx, MVSIM_EUNSUPPORTED, "%s: no kernel for this line length", what);
        if (r != 0) return cuda_fail(ctx, (cudaError_t)r, what);
        return MVSIM_OK;
    }
    int launch_x(bool inverse, const FftSize& s, const XParams& q0)
    {
        XParams q = q0;
        // rows of a later CTA prefetched into the L2 (16-byte granularity of the bulk prefetch: X % 4 == 0)
        static const int xdist = prefetch_dist(3);
        static const int xidist = prefetch_dist(3);
        if (inverse) q.prefetch_dist = ((s.n * 8) % 16 == 0 && (reinterpret_cast<uintptr_t>(q.cin) & 15) == 0) ? xidist : 0;
        else q.prefetch_dist = (!psf_phase && q.X % 4 == 0 && (reinterpret_cast<uintptr_t>(q.rin) & 15) == 0) ? xdist : 0;
        StageTimer t(ctx, psf_phase ? MVSIM_T_PSF : (inverse ? MVSIM_T_FFT_XINV : MVSIM_T_FFT_XFWD));
        return finish(fft_launch(inverse ? FFT_XINV : FFT_XFWD, lanes, s.n, &q, (unsigned)x_blocks(s, q.n_rows, inverse), 1, ctx->stream), "x pass");
    }
    int launch_strided(bool inverse, const FftSize& s, const StridedParams& q0, int n_tiles, int n_outer)
    {
        StridedParams q = q0;
        strided_fill_e32(q, s.n);
        const int threads = lanes * (s.a > s.b ? s.a : s.b);
        static const int ydist2 = prefetch_dist(2), ydist4 = prefetch_dist(4), ydist1 = prefetch_dist(1);
        const int ydist = threads <= 160 ? ydist4 : (threads <= 288 ? ydist2 : ydist1);      // resident CTAs per SM: min_blocks() in fft_group.cu
        // forward image pass over row-major rows [outer][n_src][kx_count] (in_estride == kx_count, grid = tiles x outer)
        if (!inverse && !psf_phase && ydist > 0 && q.n_peers <= 1 && !q.swap_grid && q.in_tile_global && q.in_estride == q.kx_count &&
            q.in_ostride == (long long)q.n_src * q.kx_count && q.in_tstride == lanes &&
            make_rows_tensor_map(q.in, lanes, q.kx_count, q.n_src, n_outer, q.in_tmap)) {
            q.prefetch_dist = ydist; q.grid_x = n_tiles; q.grid_y = n_outer;
        }
        static const int yidist2 = prefetch_dist(2), yidist4 = prefetch_dist(4), yidist1 = prefetch_dist(1);
        const int yidist = threads <= 160 ? yidist4 : (threads <= 288 ? yidist2 : yidist1);
        // inverse pass over tile-major input [tiles][outer][n][T] (one GPU): a CTA's input is one contiguous range
        if (inverse && yidist > 0 && q.n_peers <= 1 && !q.swap_grid && q.in_estride == lanes && q.in_ostride == (long long)s.n * lanes &&
            q.tile0 == 0 && (reinterpret_cast<uintptr_t>(q.in) & 15) == 0) {
            q.prefetch_dist = yidist; q.grid_x = n_tiles; q.grid_y = n_outer;
        }
        StageTimer t(ctx, psf_phase ? MVSIM_T_PSF : (inverse ? MVSIM_T_FFT_YINV : MVSIM_T_FFT_YFWD));
        const unsigned tiles = (unsigned)n_tiles;
        const unsigned gx = q.swap_grid ? (unsigned)n_outer : tiles, gy = q.swap_grid ? tiles : (unsigned)n_outer;
        return finish(fft_launch(inverse ? FFT_SINV : FFT_SFWD, lanes, s.n, &q, gx, gy, ctx->stream), "strided pass");
    }
    // Decimated inverse of the whole-view fused z pass (ZFusedDec in fft/line_fft.cuh): used wherever the planner's split allows it
    // and the polyphase kernel does not apply (measured 2.49 -> 2.13 ms at config 3 against ZFusedOTF).  MVSIM_OPT_Z_KERNEL = 2 (or
    // MVSIM_Z_KERNEL=2 in the environment) selects the full inverse for A/B runs.
    bool z_decimate(const FftSize& s) const
    {
        return MVSIM_PACKED_FFT != 0 && ctx->z_kernel != 2 && s.n >= kDecMinLine && s.n <= kDecMaxLine;
    }
    int launch_zfused_dec(const FftSize& s, const ZFusedParams& q0, int n_tiles, int n_outer, int inc)
    {
        ZFusedParams q = q0;
        MVSIM_TRY(get_dec_table(ctx, s.n, q.crop0, q.n_src, inc, &q.dtab));  // cached per (n, crop0, n_src, inc) in the context
        StageTimer t(ctx, MVSIM_T_FFT_ZFUSED);
        q.use_tma = (zfused_otf_tma_fits(s.b, s.a, lanes, q.k_src) && make_h_tensor_map(q.p2, lanes, n_tiles, q.k_src, n_outer, q.h_tmap)) ? 1 : 0;
        const int zthreads = lanes * (s.a > s.b ? s.a : s.b);
        static const int zdist2 = prefetch_dist(2), zdist4 = prefetch_dist(4), zdist1 = prefetch_dist(1);
        const int zdist = zthreads <= 160 ? zdist4 : (zthreads <= 288 ? zdist2 : zdist1);
        q.grid_x = n_outer; q.grid_y = n_tiles;
        q.prefetch_dist = (q.use_tma && zdist > 0 && make_h_tensor_map(q.u, lanes, n_tiles, q.zg, n_outer, q.u_tmap)) ? zdist : 0;
        return finish(fft_launch(inc == 3 ? FFT_ZFUSED_DEC3 : FFT_ZFUSED_DEC5, lanes, s.n, &q, (unsigned)n_outer, (unsigned)n_tiles, ctx->stream),
                      "fused z pass (decimated inverse)");
    }
    // Polyphase form of the whole-view fused z pass (ZFusedPoly in fft/zfused_poly.cuh).
    bool z_polyphase(const FftSize& s, int inc, int k_src) const
    {
        // (auto = the measured winner at BASELINE config 3, see kPolyphaseDefault)
        const bool want = ctx->z_kernel == 3 || (ctx->z_kernel == 0 && kPolyphaseDefault);
        if (!want || MVSIM_PACKED_FFT == 0 || s.n < kDecMinLine || s.n > kDecMaxLine) return false;
        return zfused_poly_fits(s.n, inc, lanes, k_src);
    }
    int launch_zfused_poly(const FftSize& s, const ZFusedParams& q0, int n_tiles, int n_outer, int inc)
    {
        ZFusedParams q = q0;
        if (!make_h_tensor_map(q.p2, lanes, n_tiles, q.k_src, n_outer, q.h_tmap)) return -2;      // the kernel needs the TMA-fed PSF tile
        q.use_tma = 1;
        StageTimer t(ctx, MVSIM_T_FFT_ZFUSED);
        static const int zdist2 = prefetch_dist(2);        // (half and twice this distance measured: 1.815 / 1.816 ms, the same)
        q.grid_x = n_outer; q.grid_y = n_tiles;
        q.prefetch_dist = (q.use_tma && zdist2 > 0 && make_h_tensor_map(q.u, lanes, n_tiles, q.zg, n_outer, q.u_tmap)) ? zdist2 : 0;
        return finish(fft_launch(inc == 3 ? FFT_ZFUSED_POLY3 : FFT_ZFUSED_POLY5, lanes, s.n, &q, (unsigned)n_outer, (unsigned)n_tiles, ctx->stream),
                      "fused z pass (polyphase)");
    }
    int launch_zfused(const FftSize& s, const ZFusedParams& q0, int n_tiles, int n_outer)
    {
        StageTimer t(ctx, MVSIM_T_FFT_ZFUSED);
        const unsigned tiles = (unsigned)n_tiles;
        ZFusedParams q = q0;
        if (q.h_mode) {
            // PSF tile [KZ rows] through the TMA unit into its own shared-memory area
            q.use_tma = (zfused_otf_tma_fits(s.a, s.b, lanes, q.k_src) && make_h_tensor_map(q.p2, lanes, n_tiles, q.k_src, n_outer, q.h_tmap)) ? 1 : 0;
            const int zthreads = lanes * (s.a > s.b ? s.a : s.b);
            static const int zdist2 = prefetch_dist(2), zdist4 = prefetch_dist(4), zdist1 = prefetch_dist(1);
            const int zdist = zthreads <= 160 ? zdist4 : (zthreads <= 288 ? zdist2 : zdist1);
            q.grid_x = n_outer; q.grid_y = n_tiles;
            q.prefetch_dist = (q.use_tma && zdist > 0 && q.n_peers <= 1 && q.estride32 != 0 &&
                               make_h_tensor_map(q.u, lanes, n_tiles, q.zg, n_outer, q.u_tmap)) ? zdist : 0;
            return finish(fft_launch(FFT_ZFUSED_OTF, lanes, s.n, &q, (unsigned)n_outer, tiles, ctx->stream), "fused z pass (PSF spectrum on the fly)");
        }
        q.use_tma = make_h_tensor_map(q.h, lanes, n_tiles, s.n, n_outer, q.h_tmap) ? 1 : 0;
        return finish(fft_launch(FFT_ZFUSED, lanes, s.n, &q, (unsigned)n_outer, tiles, ctx->stream), "fused z pass");
    }
};

}  // namespace

int strided_lanes() { return 8; }

// PSF-spectrum cache.  Hashes the (normalised) PSF on the device, reads the 16 bytes back (one stream synchronisation per
// convolution: ~20 us against a >= 0.28 ms PSF stage at config 3) and looks the key up.  Hit: *p2 is the cached partial spectrum.
// Miss: *p2 is a fresh cache-owned buffer the caller must fill (entries beyond the byte budget are evicted least recently used;
// the stream is idle at that point, so no kernel still reads them).  *p2 == nullptr: not cacheable (budget too small / no memory).
static int psf_cache_lookup(mvsim_ctx* ctx, const float* d_psf, const ConvPlan& pl, int lanes, size_t p2_elems, float2** p2, bool* hit)
{
    *p2 = nullptr; *hit = false;
    const size_t bytes = p2_elems * sizeof(float2);
    if (ctx->psf_cache_max_bytes == 0 || bytes > ctx->psf_cache_max_bytes) return MVSIM_OK;
    if (!ctx->d_hash) {
        MVSIM_CUDA(ctx, cudaMalloc((void**)&ctx->d_hash, 2 * sizeof(unsigned long long)));
        MVSIM_CUDA(ctx, cudaHostAlloc((void**)&ctx->h_hash, 2 * sizeof(unsigned long long), cudaHostAllocDefault));
    }
    const size_t n = (size_t)pl.kdims[0] * pl.kdims[1] * pl.kdims[2];
    MVSIM_TRY(k_hash128(ctx, d_psf, n, ctx->d_hash));
    MVSIM_CUDA(ctx, cudaMemcpyAsync(ctx->h_hash, ctx->d_hash, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    MVSIM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const std::array<uint64_t, 9> key = { ctx->h_hash[0], ctx->h_hash[1], (uint64_t)pl.kdims[0], (uint64_t)pl.kdims[1], (uint64_t)pl.kdims[2],
                                          (uint64_t)pl.sx.n, (uint64_t)pl.sy.n, (uint64_t)pl.sz.n, (uint64_t)lanes };
    const uint64_t now = ++ctx->psf_cache_tick;
    for (auto& e : ctx->psf_cache)
        if (e.key == key) { e.last_use = now; *p2 = e.p2; *hit = true; ctx->psf_cache_hits++; return MVSIM_OK; }
    ctx->psf_cache_misses++;
    size_t held = 0;
    for (auto& e : ctx->psf_cache) held += e.bytes;
    while (!ctx->psf_cache.empty() && held + bytes > ctx->psf_cache_max_bytes) {
        size_t lru = 0;
        for (size_t i = 1; i < ctx->psf_cache.size(); ++i)
            if (ctx->psf_cache[i].last_use < ctx->psf_cache[lru].last_use) lru = i;
        held -= ctx->psf_cache[lru].bytes;
        cudaFree(ctx->psf_cache[lru].p2);
        ctx->psf_cache.erase(ctx->psf_cache.begin() + (long)lru);
    }
    float2* buf = nullptr;
    if (cudaMalloc((void**)&buf, bytes) != cudaSuccess) { cudaGetLastError(); return MVSIM_OK; }      // no room: plain path
    ctx->psf_cache.push_back({ key, buf, bytes, now });
    *p2 = buf;
    return MVSIM_OK;
}

static int plan_error(mvsim_ctx* ctx, int perr)
{
    if (perr == 1) return set_error(ctx, MVSIM_EINVAL, "convolve: bad dims");
    return set_error(ctx, MVSIM_EUNSUPPORTED,
                     "convolve: unsupported size (x: X+KX-1 <= 3200, z: Z+KZ-1 <= 1600, KY <= 1600; slabs need Z and the kx tile count "
                     "divisible by the number of ranks)");
}

int conv_device(mvsim_ctx* ctx, const float* img, const int64_t dims[3], const float* psf, const int64_t kdims[3],
                float* out, double* d_sum, int keep_inc, int* out_planes)
{
    const int lanes = strided_lanes();
    ConvPlan pl;
    int perr = make_conv_plan(dims, kdims, &pl);
    if (perr) return plan_error(ctx, perr);
    SlabGeom g;
    if ((perr = make_slab_geom(pl, lanes, 0, 1, &g))) return plan_error(ctx, perr);
    mvsim_tables tx, ty, tz;
    MVSIM_TRY(get_tables(ctx, pl.sx.n, &tx));
    MVSIM_TRY(get_tables(ctx, pl.sy.n, &ty));
    MVSIM_TRY(get_tables(ctx, pl.sz.n, &tz));

    DevBufs buf(ctx);
    ConvWorkspace ws = {};
    ws.u1 = ws.u1o = buf.alloc<float2>((size_t)pl.u1_elems(g.z_local));
    if (pl.y_blocks > 1) ws.u1o = buf.alloc<float2>((size_t)pl.u1_elems(g.z_local));   // blocks still read halo rows of u1
    ws.u2 = ws.ex = buf.alloc<float2>((size_t)pl.u2_elems(lanes, g.z_local));
    if (!otf_default()) ws.h = buf.alloc<float2>((size_t)pl.h_elems(lanes, g.tiles_own));
    MVSIM_TRY(buf.st);
    // PSF partial spectrum: from the cache when this (normalised) PSF has been seen with this plan, else computed -- into a
    // cache-owned buffer when the cache is on, into a pool buffer otherwise
    bool psf_hit = false;
    float2* cached = nullptr;
    if (otf_default()) {
        StageTimer t(ctx, MVSIM_T_PSF);
        MVSIM_TRY(psf_cache_lookup(ctx, psf, pl, lanes, (size_t)pl.p2_elems(lanes, g.tiles_own), &cached, &psf_hit));
    }
    ws.p2 = cached ? cached : buf.alloc<float2>((size_t)pl.p2_elems(lanes, g.tiles_own));
    if (!psf_hit) ws.p1 = buf.alloc<float2>((size_t)pl.p1_elems());
    ws.tw_x = tx.tw; ws.twist_x = tx.twist; ws.tw_y = ty.tw; ws.tw_z = tz.tw;

    CudaLauncher l = { ctx, true, lanes };
    const int planes = conv_out_planes(pl, g, keep_inc);
    if (out_planes) *out_planes = planes;
    const int nblocks = CudaLauncher::x_blocks(pl.sx, pl.dims[1] * planes, true);      // per-block sums of the inverse x pass
    double* partials = d_sum ? buf.alloc<double>((size_t)nblocks) : nullptr;
    MVSIM_TRY(buf.st);
    if (!psf_hit) MVSIM_TRY(conv_psf_spectrum(l, pl, g, ws, psf));
    l.psf_phase = false;
    MVSIM_TRY(conv_apply(l, pl, g, ws, img, out, partials, keep_inc));
    if (d_sum) {
        StageTimer t(ctx, MVSIM_T_ADJUST);
        MVSIM_TRY(k_sum_partials(ctx, partials, (size_t)nblocks, d_sum));
    }
    return MVSIM_OK;
}

}  // namespace mvsim

// ---- slab-decomposed convolution of the largest single volume (SURVEY section 8e, BASELINE config 5) ----------------
// One plan per rank.  The exchange buffers are owned by the caller (torch tensors in the Python
// orchestrator, so torch.distributed / NCCL can run the two all-to-all transposes on them).
struct mvsim_slabconv {
    mvsim::ConvPlan pl;
    mvsim::SlabGeom g;
    int lanes;
    mvsim::ConvWorkspace ws;
    void* owned[16];
    int n_owned;
    float2 *send, *recv;
    // peer-to-peer mode: per buffer set the z-pass buffer X and the inverse-side buffer Y of every rank
    int p2p_sets;
    float2* px[2][mvsim::kMaxRanks];
    float2* py[2][mvsim::kMaxRanks];
    void* opened[4 * mvsim::kMaxRanks];
    int n_opened;
};

using namespace mvsim;

extern "C" {

int mvsim_slabconv_create(mvsim_ctx* ctx, const int64_t dims[3], const int64_t kdims[3], int rank, int world, mvsim_slabconv** out)
{
    if (!ctx || !dims || !kdims || !out) return set_error(ctx, MVSIM_EINVAL, "slabconv_create: null argument");
    *out = nullptr;
    MVSIM_ENTER(ctx);
    mvsim_slabconv* p = new mvsim_slabconv();
    p->lanes = strided_lanes();
    p->n_owned = 0;
    p->send = p->recv = nullptr;
    p->p2p_sets = 0;
    p->n_opened = 0;
    int perr = make_conv_plan(dims, kdims, &p->pl);
    if (!perr) perr = make_slab_geom(p->pl, p->lanes, rank, world, &p->g);
    if (perr) { delete p; return plan_error(ctx, perr); }
    int st = MVSIM_OK;
    mvsim_tables tx, ty, tz;
    auto grab = [&](float2** dst, size_t elems) {
        if (st != MVSIM_OK) return;
        void* q = nullptr;
        cudaError_t e = cudaMalloc(&q, (elems ? elems : 1) * sizeof(float2));
        if (e != cudaSuccess) { st = cuda_fail(ctx, e, "cudaMalloc(slabconv workspace)"); return; }
        p->owned[p->n_owned++] = q;
        *dst = static_cast<float2*>(q);
    };
    if ((st = get_tables(ctx, p->pl.sx.n, &tx)) == MVSIM_OK && (st = get_tables(ctx, p->pl.sy.n, &ty)) == MVSIM_OK &&
        (st = get_tables(ctx, p->pl.sz.n, &tz)) == MVSIM_OK) {
        p->ws = ConvWorkspace{};
        grab(&p->ws.u1, (size_t)p->pl.u1_elems(p->g.z_local));
        p->ws.u1o = p->ws.u1;
        if (p->pl.y_blocks > 1) grab(&p->ws.u1o, (size_t)p->pl.u1_elems(p->g.z_local));
        if (!otf_default()) grab(&p->ws.h, (size_t)p->pl.h_elems(p->lanes, p->g.tiles_own));
        grab(&p->ws.p1, (size_t)p->pl.p1_elems());
        grab(&p->ws.p2, (size_t)p->pl.p2_elems(p->lanes, p->g.tiles_own));
        p->ws.tw_x = tx.tw; p->ws.twist_x = tx.twist; p->ws.tw_y = ty.tw; p->ws.tw_z = tz.tw;
    }
    if (st != MVSIM_OK) {
        for (int i = 0; i < p->n_owned; ++i) cudaFree(p->owned[i]);
        delete p;
        return st;
    }
    *out = p;
    return MVSIM_OK;
}

int mvsim_slabconv_destroy(mvsim_ctx* ctx, mvsim_slabconv* p)
{
    if (!p) return MVSIM_OK;
    DeviceScope scope(ctx ? ctx->device : 0);
    if (ctx) cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < p->n_opened; ++i) cudaIpcCloseMemHandle(p->opened[i]);
    for (int i = 0; i < p->n_owned; ++i) cudaFree(p->owned[i]);
    delete p;
    return MVSIM_OK;
}

// ---- peer-to-peer mode: the exchanges are fused into the y forward pass and the fused z pass (NVLink stores) ----------
int mvsim_slabconv_p2p_alloc(mvsim_ctx* ctx, mvsim_slabconv* p, int nbuf, unsigned char* handles_out)
{
    if (!ctx || !p || !handles_out || nbuf < 1 || nbuf > 2) return set_error(ctx, MVSIM_EINVAL, "slabconv_p2p_alloc: bad argument");
    if (p->g.world > kMaxRanks) return set_error(ctx, MVSIM_EUNSUPPORTED, "slabconv_p2p: at most %d ranks", kMaxRanks);
    if (p->p2p_sets) return set_error(ctx, MVSIM_EINVAL, "slabconv_p2p_alloc: already allocated");
    MVSIM_ENTER(ctx);
    const size_t bytes = (size_t)p->pl.u2_elems(p->lanes, p->g.z_local) * sizeof(float2);
    for (int i = 0; i < nbuf; ++i)
        for (int k = 0; k < 2; ++k) {
            void* q = nullptr;
            MVSIM_CUDA(ctx, cudaMalloc(&q, bytes));
            p->owned[p->n_owned++] = q;
            (k == 0 ? p->px : p->py)[i][p->g.rank] = static_cast<float2*>(q);
            cudaIpcMemHandle_t h;
            MVSIM_CUDA(ctx, cudaIpcGetMemHandle(&h, q));
            static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t size");
            memcpy(handles_out + (size_t)(i * 2 + k) * 64, &h, 64);
        }
    p->p2p_sets = nbuf;
    return MVSIM_OK;
}

int mvsim_slabconv_p2p_open(mvsim_ctx* ctx, mvsim_slabconv* p, const unsigned char* all_handles)
{
    if (!ctx || !p || !all_handles || !p->p2p_sets) return set_error(ctx, MVSIM_EINVAL, "slabconv_p2p_open: allocate first");
    MVSIM_ENTER(ctx);
    const int per_rank = p->p2p_sets * 2;
    for (int r = 0; r < p->g.world; ++r) {
        if (r == p->g.rank) continue;
        for (int i = 0; i < p->p2p_sets; ++i)
            for (int k = 0; k < 2; ++k) {
                cudaIpcMemHandle_t h;
                memcpy(&h, all_handles + ((size_t)r * per_rank + i * 2 + k) * 64, 64);
                void* q = nullptr;
                MVSIM_CUDA(ctx, cudaIpcOpenMemHandle(&q, h, cudaIpcMemLazyEnablePeerAccess));
                p->opened[p->n_opened++] = q;
                (k == 0 ? p->px : p->py)[i][r] = static_cast<float2*>(q);
            }
    }
    return MVSIM_OK;
}

int mvsim_slabconv_p2p_select(mvsim_slabconv* p, int set)
{
    if (!p || set < 0 || set >= p->p2p_sets) return MVSIM_EINVAL;
    p->ws.n_peers = p->g.world;
    for (int r = 0; r < p->g.world; ++r) { p->ws.peers_x[r] = p->px[set][r]; p->ws.peers_y[r] = p->py[set][r]; }
    p->send = p->py[set][p->g.rank];
    p->recv = p->px[set][p->g.rank];
    p->ws.u2 = p->send;         // the inverse y pass reads what the peers' z passes delivered
    p->ws.ex = p->recv;         // the fused z pass reads what the peers' y passes delivered
    return MVSIM_OK;
}

int mvsim_slabconv_info(const mvsim_slabconv* p, int64_t info[8])
{
    if (!p || !info) return MVSIM_EINVAL;
    info[0] = p->g.z_local; info[1] = p->g.z0; info[2] = p->pl.y_blocks;
    info[3] = p->pl.u2_elems(p->lanes, p->g.z_local);         // float2 elements of each exchange buffer
    info[4] = 2 * p->pl.sx.n; info[5] = p->pl.sy.n; info[6] = p->pl.sz.n;
    info[7] = p->g.tiles_own;
    return MVSIM_OK;
}

int mvsim_slabconv_bind(mvsim_slabconv* p, void* send_buffer, void* recv_buffer)
{
    if (!p || !send_buffer || (p->g.world > 1 && !recv_buffer)) return MVSIM_EINVAL;
    p->send = static_cast<float2*>(send_buffer);
    p->recv = p->g.world > 1 ? static_cast<float2*>(recv_buffer) : p->send;
    p->ws.u2 = p->send;
    p->ws.ex = p->recv;
    return MVSIM_OK;
}

#define MVSIM_SLAB_ENTER(ctx, p)                                                                   \
    if (!(ctx) || !(p)) return mvsim::set_error((ctx), MVSIM_EINVAL, "slabconv: null argument");   \
    if (!(p)->send) return mvsim::set_error((ctx), MVSIM_EINVAL, "slabconv: bind the exchange buffers first"); \
    MVSIM_ENTER(ctx)

int mvsim_slabconv_prepare(mvsim_ctx* ctx, mvsim_slabconv* p, const float* d_psf, const float* d_img_slab)
{
    MVSIM_SLAB_ENTER(ctx, p);
    if (!d_psf || !d_img_slab) return set_error(ctx, MVSIM_EINVAL, "slabconv_prepare: null buffer");
    CudaLauncher l = { ctx, true, p->lanes };
    MVSIM_TRY(conv_psf_spectrum(l, p->pl, p->g, p->ws, d_psf));
    l.psf_phase = false;
    return conv_forward_x(l, p->pl, p->g, p->ws, d_img_slab);
}

int mvsim_slabconv_forward_y(mvsim_ctx* ctx, mvsim_slabconv* p, int block)
{
    MVSIM_SLAB_ENTER(ctx, p);
    if (block < 0 || block >= p->pl.y_blocks) return set_error(ctx, MVSIM_EINVAL, "slabconv: bad block");
    CudaLauncher l = { ctx, false, p->lanes };
    return conv_forward_y(l, p->pl, p->g, p->ws, block);
}

int mvsim_slabconv_middle_z(mvsim_ctx* ctx, mvsim_slabconv* p)
{
    MVSIM_SLAB_ENTER(ctx, p);
    CudaLauncher l = { ctx, false, p->lanes };
    return conv_middle_z(l, p->pl, p->g, p->ws, p->ws.ex, 1);
}

int mvsim_slabconv_inverse_y(mvsim_ctx* ctx, mvsim_slabconv* p, int block)
{
    MVSIM_SLAB_ENTER(ctx, p);
    if (block < 0 || block >= p->pl.y_blocks) return set_error(ctx, MVSIM_EINVAL, "slabconv: bad block");
    CudaLauncher l = { ctx, false, p->lanes };
    return conv_inverse_y(l, p->pl, p->g, p->ws, block, p->g.z_local);
}

int mvsim_slabconv_finish(mvsim_ctx* ctx, mvsim_slabconv* p, float* d_out_slab)
{
    MVSIM_SLAB_ENTER(ctx, p);
    if (!d_out_slab) return set_error(ctx, MVSIM_EINVAL, "slabconv_finish: null buffer");
    CudaLauncher l = { ctx, false, p->lanes };
    return conv_inverse_x(l, p->pl, p->ws, d_out_slab, nullptr, p->g.z_local);
}

}  // extern "C"
