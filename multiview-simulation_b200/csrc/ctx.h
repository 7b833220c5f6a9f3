// Context of libmvsim.so: device, stream, error text, cached tables, event profiling.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <array>
#include <map>
#include <string>
#include <vector>

#include "../../include/mvsim.h"

struct mvsim_volume {
    float* d;
    int64_t dims[3];
    int device;
    bool borrowed = false;      // mvsim_volume_wrap: memory owned by the caller (e.g. a torch tensor filled by an NCCL broadcast)
    size_t elems() const { return (size_t)(dims[0] * dims[1] * dims[2]); }
};

struct mvsim_tables { float2 *tw, *twist; };

struct mvsim_ctx {
    int device;
    cudaStream_t stream;
    bool own_stream;
    cudaStream_t copy_stream;                // lazily created: result downloads overlapping the next view
    cudaMemPool_t mempool;                   // this context's own stream-ordered pool: workspaces are never traded between
                                             // the streams of two contexts (callers run contexts concurrently)
    std::string err;
    double* d_scalars;                       // [8] device doubles: sums, corrections
    std::map<int, mvsim_tables> tables;      // by complex line length
    std::map<std::array<int, 4>, float2*> dec_tables;   // decimated fused z pass: D' table by (n, crop0, n_src, inc)
    // PSF-spectrum cache (SURVEY C6): partial spectra P2 keyed by a device-computed content hash of the NORMALISED PSF + the plan.
    // The reference rebuilds the kernel FFT on every call (S/SimulateMultiViewDataset.java:257) although its callers reuse one
    // PSF across SNR sweeps and tile pairs (S/SimulateTileStitching.java:71,95,110); results are bit-identical either way.
    struct PsfEntry { std::array<uint64_t, 9> key; float2* p2; size_t bytes; uint64_t last_use; };
    std::vector<PsfEntry> psf_cache;
    size_t psf_cache_max_bytes;              // 0 = off
    uint64_t psf_cache_tick, psf_cache_hits, psf_cache_misses;
    unsigned long long* d_hash;              // [2] device words
    unsigned long long* h_hash;              // [2] pinned host words
    // count transport of the batch call (MVSIM_OPT_COUNT_TRANSPORT): Poisson counts cross the host link as uint16 and are widened to
    // the float32 of the reference's API by host threads inside the call
    int count_transport;                     // 0 = float32 (default), 1 = uint16 when snr >= 0
    int host_threads;                        // widening threads (0 = default)
    int z_kernel;                            // MVSIM_OPT_Z_KERNEL: 0 auto, 1 no polyphase kernel, 2 full spectral kernel only
    struct Staging { void* p; size_t bytes; };
    std::vector<Staging> staging;            // pinned uint16 staging buffers, kept across calls
    void* widen_pool;                        // mvsim::WidenPool*, lazily created
    int64_t launches;
    // profiling
    bool profiling;
    struct Ev { cudaEvent_t a, b; int stage; };
    std::vector<Ev> events;                  // recorded since last reset
    std::vector<Ev> pool;                    // reusable
    double acc_ms[MVSIM_NSTAGES];
    int64_t acc_n[MVSIM_NSTAGES];
};

namespace mvsim {

int set_error(mvsim_ctx* ctx, int status, const char* fmt, ...);
int cuda_fail(mvsim_ctx* ctx, cudaError_t e, const char* what);

#define MVSIM_CUDA(ctx, call)                                             \
    do {                                                                  \
        cudaError_t e__ = (call);                                         \
        if (e__ != cudaSuccess) return mvsim::cuda_fail((ctx), e__, #call); \
    } while (0)
#define MVSIM_TRY(call)                    \
    do {                                   \
        int s__ = (call);                  \
        if (s__ != MVSIM_OK) return s__;   \
    } while (0)

// Every exported function that touches a device runs inside one of these: it makes `device` current (ok tells whether that
// worked) and gives the caller's current device back on exit.  It also drops a stale, non-sticky error an earlier call of this
// host thread left behind (ours or the caller's): the launch checks of the entry point read cudaGetLastError() and must report
// their own failures only.
struct DeviceScope {
    int prev = -1;
    bool ok = false;
    explicit DeviceScope(int device)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; return; }
        ok = cudaSetDevice(device) == cudaSuccess;
        if (ok) cudaGetLastError();
    }
    ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
};

#define MVSIM_ENTER(ctx)                                                                     \
    if (!(ctx)) return mvsim::set_error(nullptr, MVSIM_EINVAL, "null context");             \
    mvsim::DeviceScope scope__((ctx)->device);                                               \
    if (!scope__.ok) return mvsim::set_error((ctx), MVSIM_ECUDA, "cannot select CUDA device %d", (ctx)->device)

// RAII-less scoped stage timer: begin() before the launches of a stage, end() after.
struct StageTimer {
    mvsim_ctx* ctx; int idx;
    StageTimer(mvsim_ctx* c, int stage);
    ~StageTimer();
};

int dev_alloc(mvsim_ctx* ctx, void** p, size_t bytes);      // stream-ordered (cudaMallocAsync)
void dev_free(mvsim_ctx* ctx, void* p);
int get_tables(mvsim_ctx* ctx, int n, mvsim_tables* t);

// device buffers of one call with a deferred failure: after the first failed allocation alloc() returns null and st keeps that
// status, so a call allocates all it needs and checks once
struct DevBufs {
    mvsim_ctx* ctx;
    int st = MVSIM_OK;
    std::vector<void*> held;
    explicit DevBufs(mvsim_ctx* c) : ctx(c) {}
    ~DevBufs() { free_all(); }
    template <class T> T* alloc(size_t n)
    {
        void* q = nullptr;
        if (st == MVSIM_OK && (st = dev_alloc(ctx, &q, n * sizeof(T))) == MVSIM_OK) held.push_back(q);
        return static_cast<T*>(q);
    }
    void free_all() { for (void* q : held) dev_free(ctx, q); held.clear(); }
};

// stage kernels (stages.cu); all enqueue on ctx->stream
int k_rotate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], int axis, const double inv[12]);
// fused; MVSIM_EUNSUPPORTED when the rotation is not the axis-0 fast path.  z_local > 0: only the output planes [z0, z0 + z_local)
// of the view (out = that slab), the source `in` stays the whole volume
int k_rotate_attenuate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], int axis, const double inv[12], double delta,
                       int steps, int64_t z0 = 0, int64_t z_local = 0);
int k_attenuate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], double delta, int steps);
int k_sum(mvsim_ctx* ctx, const float* in, size_t n, double* d_sum);                 // deterministic double sum
int k_sum_partials(mvsim_ctx* ctx, const double* partials, size_t n, double* d_sum);
int k_divide_by_sum(mvsim_ctx* ctx, float* inout, size_t n, const double* d_sum);     // (float)((double)v / sum)
int k_adjust_corr(mvsim_ctx* ctx, const double* d_sum, size_t n, float min_value, float target_avg, double* d_corr);
int k_adjust_apply(mvsim_ctx* ctx, float* inout, size_t n, const double* d_corr, float min_value);
int k_adjust_corr_ranks(mvsim_ctx* ctx, const double* d_sums, int world, double n_global, float min_value, float target_avg, double* d_corr);
int k_extract_slab(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int64_t z0, int64_t z_local, int inc, const double* d_corr,
                   float min_value, float snr, uint64_t seed, uint64_t stream, float* out, int64_t* planes_out, unsigned short* out16 = nullptr,
                   int* d_overflow = nullptr);
// k_extract that also writes the counts as uint16 (count transport of the batch call) and ORs *d_overflow when one exceeds 65535
int k_extract_u16(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, const double* d_corr, float min_value,
                  float snr, uint64_t seed, uint64_t stream, float* out, unsigned short* out16, int* d_overflow);
// out[x,y,cz] = f(in[x,y,cz*inc]); d_corr != null fuses adjustImage; snr >= 0 adds Poisson noise
int k_extract(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, const double* d_corr, float min_value,
              float snr, uint64_t seed, uint64_t stream, float* out);
// k_extract of the dense cut [min, max] (inclusive, x y z) of `in`, read in place; the bounds are the caller's to check
int k_extract_interval(mvsim_ctx* ctx, const float* in, const int64_t dims[3], const int64_t min[3], const int64_t max[3], int inc,
                       float snr, uint64_t seed, uint64_t stream, float* out);
int k_make_isotropic(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, float* out);
int k_weight_image(mvsim_ctx* ctx, const int64_t dims[3], float* out);
int k_normalize_weights(mvsim_ctx* ctx, float* const* d_weights, int n_views, size_t n, float osem, float* d_sum_out);
// rotateAroundAxis(makeIsotropic(acq, inc), 0, .) straight from the acquired planes; acq_dims = {X, Y, Za}, out: X*Y*((Za-1)*inc+1);
// inv = axisRotation(iso dims, 0, degrees) inverse
int k_align_view(mvsim_ctx* ctx, const float* acq, const int64_t acq_dims[3], int inc, const double inv[12], float* out);
// normalised rotate-back weights of n_all views (inv: n_all x 12, the axis-0 inverses for dims): view views[j] -> outs[j] (j < n_out),
// the sum of the normalised weights -> sum_out (nullable); no input volume
int k_aligned_weights(mvsim_ctx* ctx, const int64_t dims[3], int n_all, const double* inv, float osem, int n_out, const int* views,
                      float* const* outs, float* sum_out);
int k_poisson(mvsim_ctx* ctx, float* inout, size_t n, double snr, uint64_t seed, uint64_t stream);
// 128-bit content hash of n floats (order-independent sum of two 64-bit mixes of (bits, index)): d_out[2], enqueued on the stream
int k_hash128(mvsim_ctx* ctx, const float* in, size_t n, unsigned long long* d_out);

// input generators (phantom.cu).  points / host_rec / host_val are HOST arrays (consumed before return), the rest device pointers
int k_render_beads(mvsim_ctx* ctx, const double* points, int n, const double sigma[3], const int64_t imin[3], const int64_t imax[3], float* d_out);
int k_paint_spheres(mvsim_ctx* ctx, float* d_img, const int64_t dims[3], const int* host_rec /* n x (cx, cy, cz, radius) */, const float* host_val, int n);
int k_downsample2x(mvsim_ctx* ctx, const float* in, const int64_t dims[3], float* out);
int k_make_square(mvsim_ctx* ctx, const float* in, const int64_t dims[3], float* out);

// convolution driver (conv.cu): psf normalised, device pointers; sum of the output voxels -> d_sum when non-null.
// keep_inc > 1: out receives *out_planes planes -- the slices z = 0, inc, ... and one plane with the sum of the rest
// (see conv_out_planes in fft/conv_driver.h); d_sum is still the sum over the whole convolved volume.
int conv_device(mvsim_ctx* ctx, const float* img, const int64_t dims[3], const float* psf, const int64_t kdims[3],
                float* out, double* d_sum, int keep_inc = 1, int* out_planes = nullptr);

}  // namespace mvsim
