// C ABI of libmvsim.so (include/mvsim.h).  Host-side orchestration only; kernels live in stages.cu
// and fft/.  There is deliberately no CPU path: without a CUDA device every compute call fails.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <stdlib.h>
#include <thread>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include "ctx.h"
#include "fft/conv_plan.h"

namespace mvsim {

static thread_local std::string tls_error;

int set_error(mvsim_ctx* ctx, int status, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    tls_error = buf;
    if (ctx) ctx->err = buf;
    return status;
}

int cuda_fail(mvsim_ctx* ctx, cudaError_t e, const char* what)
{
    return set_error(ctx, e == cudaErrorMemoryAllocation ? MVSIM_ENOMEM : MVSIM_ECUDA, "CUDA error %d (%s) in %s", (int)e,
                     cudaGetErrorString(e), what);
}

StageTimer::StageTimer(mvsim_ctx* c, int stage) : ctx(c), idx(-1)
{
    if (!c->profiling) return;
    mvsim_ctx::Ev ev;
    if (!c->pool.empty()) { ev = c->pool.back(); c->pool.pop_back(); }
    else if (cudaEventCreate(&ev.a) != cudaSuccess || cudaEventCreate(&ev.b) != cudaSuccess) return;
    ev.stage = stage;
    cudaEventRecord(ev.a, c->stream);
    c->events.push_back(ev);
    idx = (int)c->events.size() - 1;
}

StageTimer::~StageTimer()
{
    if (idx >= 0) cudaEventRecord(ctx->events[idx].b, ctx->stream);
}

int dev_alloc(mvsim_ctx* ctx, void** p, size_t bytes)
{
    if (bytes == 0) bytes = 16;
    cudaError_t e = ctx->mempool ? cudaMallocFromPoolAsync(p, bytes, ctx->mempool, ctx->stream) : cudaMallocAsync(p, bytes, ctx->stream);
    if (e != cudaSuccess) { *p = nullptr; return cuda_fail(ctx, e, "cudaMallocAsync"); }
    return MVSIM_OK;
}

void dev_free(mvsim_ctx* ctx, void* p)
{
    if (p) cudaFreeAsync(p, ctx->stream);
}

int get_tables(mvsim_ctx* ctx, int n, mvsim_tables* t)
{
    auto it = ctx->tables.find(n);
    if (it != ctx->tables.end()) { *t = it->second; return MVSIM_OK; }
    std::vector<float> host((size_t)4 * n);
    fill_twiddles(n, host.data());
    fill_twist(n, host.data() + 2 * n);
    float2* d = nullptr;
    MVSIM_CUDA(ctx, cudaMalloc((void**)&d, sizeof(float2) * 2 * n));
    // synchronous copy from pageable memory: the host vector may die right after
    MVSIM_CUDA(ctx, cudaMemcpy(d, host.data(), sizeof(float2) * 2 * n, cudaMemcpyHostToDevice));
    mvsim_tables nt = { d, d + n };
    ctx->tables[n] = nt;
    *t = nt;
    return MVSIM_OK;
}

// axisRotation S/SimulateMultiViewDataset.java:80-102 and mpicbg AffineModel3D.createInverse()
static void preconcat(double* t, const double* a)
{
    double r[12];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) r[4 * i + j] = a[4 * i] * t[j] + a[4 * i + 1] * t[4 + j] + a[4 * i + 2] * t[8 + j];
        r[4 * i + 3] = a[4 * i] * t[3] + a[4 * i + 1] * t[7] + a[4 * i + 2] * t[11] + a[4 * i + 3];
    }
    memcpy(t, r, sizeof(r));
}

static int axis_rotation(const int64_t dims[3], int axis, int degrees, double fwd[12], double inv[12])
{
    if (axis < 0 || axis > 2) return MVSIM_EINVAL;
    double c[3];
    for (int d = 0; d < 3; ++d) c[d] = (double)((dims[d] - 1) / 2);            // (max - min) / 2, long division
    const double th = (double)(float)((double)degrees / 180.0 * 3.14159265358979323846);   // (float)Math.toRadians
    const double cs = cos(th), sn = sin(th);
    double rot[12] = { 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0 };
    if (axis == 0) { rot[5] = cs; rot[6] = -sn; rot[9] = sn; rot[10] = cs; }
    else if (axis == 1) { rot[0] = cs; rot[2] = sn; rot[8] = -sn; rot[10] = cs; }
    else { rot[0] = cs; rot[1] = -sn; rot[4] = sn; rot[5] = cs; }
    const double t1[12] = { 1, 0, 0, -c[0], 0, 1, 0, -c[1], 0, 0, 1, -c[2] };
    const double t2[12] = { 1, 0, 0, c[0], 0, 1, 0, c[1], 0, 0, 1, c[2] };
    double m[12];
    memcpy(m, t1, sizeof(m));
    preconcat(m, rot);
    preconcat(m, t2);
    const double det = m[0] * m[5] * m[10] + m[4] * m[9] * m[2] + m[8] * m[1] * m[6] - m[2] * m[5] * m[8] - m[6] * m[9] * m[0] - m[10] * m[1] * m[4];
    if (det == 0) return MVSIM_EINVAL;
    const double id = 1.0 / det;
    double i[12];
    i[0] = (m[5] * m[10] - m[6] * m[9]) * id;  i[1] = (m[2] * m[9] - m[1] * m[10]) * id;  i[2] = (m[1] * m[6] - m[2] * m[5]) * id;
    i[4] = (m[6] * m[8] - m[4] * m[10]) * id;  i[5] = (m[0] * m[10] - m[2] * m[8]) * id;  i[6] = (m[2] * m[4] - m[0] * m[6]) * id;
    i[8] = (m[4] * m[9] - m[5] * m[8]) * id;   i[9] = (m[1] * m[8] - m[0] * m[9]) * id;   i[10] = (m[0] * m[5] - m[1] * m[4]) * id;
    i[3] = -i[0] * m[3] - i[1] * m[7] - i[2] * m[11];
    i[7] = -i[4] * m[3] - i[5] * m[7] - i[6] * m[11];
    i[11] = -i[8] * m[3] - i[9] * m[7] - i[10] * m[11];
    if (fwd) memcpy(fwd, m, sizeof(m));
    if (inv) memcpy(inv, i, sizeof(i));
    return MVSIM_OK;
}

static int check_dims(mvsim_ctx* ctx, const int64_t d[3], const char* what)
{
    if (!d || d[0] < 1 || d[1] < 1 || d[2] < 1) return set_error(ctx, MVSIM_EINVAL, "%s: dims must be >= 1", what);
    if (d[0] > 0x7fffffff || d[1] > 0x7fffffff || d[2] > 0x7fffffff || (double)d[0] * (double)d[1] * (double)d[2] > 1.0e11)
        return set_error(ctx, MVSIM_EINVAL, "%s: dims too large", what);
    return MVSIM_OK;
}

static size_t elems(const int64_t d[3]) { return (size_t)(d[0] * d[1] * d[2]); }

static int attenuate_steps(mvsim_ctx* ctx, const int64_t d[3], int strict, int* steps)
{
    if (strict && d[0] > d[1])
        return set_error(ctx, MVSIM_EINVAL, "attenuate: strict_reference needs X <= Y (the reference loop bound is dimension(0) and walks out of bounds otherwise)");
    *steps = (int)(strict ? d[0] : d[1]);
    return MVSIM_OK;
}

static int h2d(mvsim_ctx* ctx, void* d, const void* h, size_t bytes)
{
    StageTimer t(ctx, MVSIM_T_H2D);
    MVSIM_CUDA(ctx, cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return MVSIM_OK;
}

static int d2h(mvsim_ctx* ctx, void* h, const void* d, size_t bytes)
{
    StageTimer t(ctx, MVSIM_T_D2H);
    MVSIM_CUDA(ctx, cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return MVSIM_OK;
}

static int sync(mvsim_ctx* ctx)
{
    MVSIM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MVSIM_OK;
}

// d_scalars[slot] -> *out, enqueued: valid after the next synchronisation of the stream
static int fetch_scalar(mvsim_ctx* ctx, int slot, double* out)
{
    MVSIM_CUDA(ctx, cudaMemcpyAsync(out, ctx->d_scalars + slot, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    return MVSIM_OK;
}

static int read_scalar(mvsim_ctx* ctx, int slot, double* out)
{
    MVSIM_TRY(fetch_scalar(ctx, slot, out));
    return sync(ctx);
}

// The staging of a host-buffer entry point: in() / out() / inout() allocate a device buffer for n floats of a host buffer at
// once; run(body) then uploads the in / inout buffers, runs body(), downloads the out / inout buffers and the scalar() slots,
// and synchronises the stream once.  A failure skips the later steps (the synchronisation still runs) and run() returns it.
class HostCall : public DevBufs {
public:
    explicit HostCall(mvsim_ctx* c) : DevBufs(c) {}
    float* in(const float* host, size_t n) { return stage(const_cast<float*>(host), n, true, false); }
    float* out(float* host, size_t n) { return stage(host, n, false, true); }
    float* inout(float* host, size_t n) { return stage(host, n, true, true); }
    void scalar(int slot, double* host) { if (host) scalars_.push_back({ slot, host }); }

    template <class Body> int run(Body body)
    {
        int s = st;
        for (const Copy& c : copies_) if (s == MVSIM_OK && c.up) s = h2d(ctx, c.dev, c.host, c.bytes);
        if (s == MVSIM_OK) s = body();
        for (const Copy& c : copies_) if (s == MVSIM_OK && c.down) s = d2h(ctx, c.host, c.dev, c.bytes);
        for (const auto& sc : scalars_) if (s == MVSIM_OK) s = fetch_scalar(ctx, sc.first, sc.second);
        const int s2 = sync(ctx);
        return s != MVSIM_OK ? s : s2;
    }

private:
    struct Copy { float* dev; float* host; size_t bytes; bool up, down; };
    float* stage(float* host, size_t n, bool up, bool down)
    {
        float* d = alloc<float>(n);
        copies_.push_back({ d, host, n * sizeof(float), up, down });
        return d;
    }
    std::vector<Copy> copies_;
    std::vector<std::pair<int, double*>> scalars_;
};

// planes z = 0, inc, 2 inc, ... that the sampler keeps of a view of dims, and the voxels they hold
static int64_t kept_planes(const int64_t dims[3], int inc) { return (dims[2] - 1) / inc + 1; }
static size_t kept_elems(const int64_t dims[3], int inc) { return (size_t)(dims[0] * dims[1] * kept_planes(dims, inc)); }

// ---- host side of the uint16 count transport ------------------------------------------------------------------------
// uint16 -> float32, streaming stores (the destination is written once and not read back by these threads)
#if defined(__x86_64__)
__attribute__((target("avx2"))) static void widen_avx2(const unsigned short* src, float* dst, size_t n)
{
    size_t i = 0;
    while (i < n && (reinterpret_cast<uintptr_t>(dst + i) & 31)) { dst[i] = (float)src[i]; ++i; }
    for (; i + 16 <= n; i += 16) {
        const __m256i v = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src + i));
        _mm256_stream_ps(dst + i, _mm256_cvtepi32_ps(_mm256_cvtepu16_epi32(_mm256_castsi256_si128(v))));
        _mm256_stream_ps(dst + i + 8, _mm256_cvtepi32_ps(_mm256_cvtepu16_epi32(_mm256_extracti128_si256(v, 1))));
    }
    for (; i < n; ++i) dst[i] = (float)src[i];
    _mm_sfence();
}
#endif
static void widen_range(const unsigned short* src, float* dst, size_t n)
{
#if defined(__x86_64__)
    static const bool avx2 = __builtin_cpu_supports("avx2");
    if (avx2) { widen_avx2(src, dst, n); return; }
#endif
    for (size_t i = 0; i < n; ++i) dst[i] = (float)src[i];
}

// a few persistent threads per context; run() splits one view over them (and the caller) and returns when it is done
class WidenPool {
public:
    explicit WidenPool(int threads) : stop_(false), job_(0), pending_(0)
    {
        for (int t = 0; t < threads; ++t) workers_.emplace_back([this, t] { loop(t); });
    }
    ~WidenPool()
    {
        { std::lock_guard<std::mutex> lk(m_); stop_ = true; }
        cv_.notify_all();
        for (auto& w : workers_) w.join();
    }
    void run(const unsigned short* src, float* dst, size_t n)
    {
        const size_t parts = workers_.size() + 1;
        const size_t chunk = ((n + parts - 1) / parts + 63) / 64 * 64;
        {
            std::lock_guard<std::mutex> lk(m_);
            src_ = src; dst_ = dst; n_ = n; chunk_ = chunk;
            pending_ = (int)workers_.size();
            ++job_;
        }
        cv_.notify_all();
        const size_t a = workers_.size() * chunk;               // the caller takes the last part
        if (a < n) widen_range(src + a, dst + a, n - a);
        std::unique_lock<std::mutex> lk(m_);
        done_.wait(lk, [this] { return pending_ == 0; });
    }
private:
    void loop(int t)
    {
        unsigned long long seen = 0;
        for (;;) {
            const unsigned short* src; float* dst; size_t n, chunk;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return stop_ || job_ != seen; });
                if (stop_) return;
                seen = job_; src = src_; dst = dst_; n = n_; chunk = chunk_;
            }
            const size_t a = (size_t)t * chunk, b = a + chunk < n ? a + chunk : n;
            if (a < n) widen_range(src + a, dst + a, b - a);
            {
                std::lock_guard<std::mutex> lk(m_);
                if (--pending_ == 0) done_.notify_all();
            }
        }
    }
    std::vector<std::thread> workers_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    bool stop_;
    unsigned long long job_;
    int pending_;
    const unsigned short* src_ = nullptr;
    float* dst_ = nullptr;
    size_t n_ = 0, chunk_ = 0;
};

static WidenPool* widen_pool(mvsim_ctx* ctx)
{
    if (!ctx->widen_pool) {
        int t = ctx->host_threads;
        if (t <= 0) {
            const unsigned hw = std::thread::hardware_concurrency();
            t = hw >= 8 ? 4 : (hw >= 4 ? 2 : 1);       // measured (profiles/r02_notes.md): 4 threads per context beat 2 and 8
        }
        ctx->widen_pool = new WidenPool(t > 1 ? t - 1 : 0);      // the calling thread is one of the t
    }
    return static_cast<WidenPool*>(ctx->widen_pool);
}

// pinned staging buffer #i of at least `bytes` (kept across calls: cudaHostAlloc of 200 MB costs tens of milliseconds)
static int staging_buffer(mvsim_ctx* ctx, size_t i, size_t bytes, void** out)
{
    if (ctx->staging.size() <= i) ctx->staging.resize(i + 1, { nullptr, 0 });
    auto& s = ctx->staging[i];
    if (s.bytes < bytes) {
        if (s.p) cudaFreeHost(s.p);
        s.p = nullptr; s.bytes = 0;
        MVSIM_CUDA(ctx, cudaHostAlloc(&s.p, bytes, cudaHostAllocDefault));
        s.bytes = bytes;
    }
    *out = s.p;
    return MVSIM_OK;
}

// ---- device-level building blocks ---------------------------------------------------------
static int dev_rotate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], int axis, int degrees)
{
    double inv[12];
    if (axis_rotation(dims, axis, degrees, nullptr, inv)) return set_error(ctx, MVSIM_EINVAL, "rotate: axis must be 0, 1 or 2");
    StageTimer t(ctx, MVSIM_T_ROTATE);
    return k_rotate(ctx, in, out, dims, axis, inv);
}

static int dev_attenuate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], double delta, int strict)
{
    int steps = 0;
    MVSIM_TRY(attenuate_steps(ctx, dims, strict, &steps));
    StageTimer t(ctx, MVSIM_T_ATTENUATE);
    return k_attenuate(ctx, in, out, dims, delta, steps);
}

static int dev_psf_normalize(mvsim_ctx* ctx, float* psf, size_t n)
{
    StageTimer t(ctx, MVSIM_T_PSF);
    MVSIM_TRY(k_sum(ctx, psf, n, ctx->d_scalars + 0));
    return k_divide_by_sum(ctx, psf, n, ctx->d_scalars + 0);
}

static int dev_adjust(mvsim_ctx* ctx, float* img, size_t n, float min_value, float target_avg)
{
    StageTimer t(ctx, MVSIM_T_ADJUST);
    MVSIM_TRY(k_sum(ctx, img, n, ctx->d_scalars + 1));
    MVSIM_TRY(k_adjust_corr(ctx, ctx->d_scalars + 1, n, min_value, target_avg, ctx->d_scalars + 2));
    return k_adjust_apply(ctx, img, n, ctx->d_scalars + 2, min_value);
}

static int check_view(mvsim_ctx* ctx, const mvsim_view_params* p)
{
    if (!p) return set_error(ctx, MVSIM_EINVAL, "null view params");
    MVSIM_TRY(check_dims(ctx, p->dims, "simulate_view dims"));
    MVSIM_TRY(check_dims(ctx, p->kdims, "simulate_view kdims"));
    if (p->inc < 1) return set_error(ctx, MVSIM_EINVAL, "simulate_view: inc must be >= 1");
    if (p->axis < 0 || p->axis > 2) return set_error(ctx, MVSIM_EINVAL, "simulate_view: axis must be 0, 1 or 2");
    return MVSIM_OK;
}

// dims and plane step of extractSlices and makeIsotropic
static int check_sampling(mvsim_ctx* ctx, const int64_t dims[3], int inc, const char* what)
{
    MVSIM_TRY(check_dims(ctx, dims, what));
    if (inc < 1) return set_error(ctx, MVSIM_EINVAL, "%s: inc must be >= 1", what);
    return MVSIM_OK;
}

static int dev_extract_slices(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, float snr, uint64_t seed, uint64_t stream,
                              float* out)
{
    StageTimer t(ctx, MVSIM_T_SAMPLE);
    return k_extract(ctx, in, dims, inc, nullptr, 0.f, snr, seed, stream, out);
}

// rotate (axis: the caller's to check) and attenuate in one pass; MVSIM_EUNSUPPORTED, without an error text, when the rotation
// is not the axis-0 fast path.  z_local > 0: only the output planes [z0, z0 + z_local) (out = that slab)
static int dev_rotate_attenuate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], int axis, int degrees, double delta,
                                int strict, int64_t z0 = 0, int64_t z_local = 0)
{
    double inv[12];
    int steps = 0;
    axis_rotation(dims, axis, degrees, nullptr, inv);
    MVSIM_TRY(attenuate_steps(ctx, dims, strict, &steps));
    StageTimer t(ctx, MVSIM_T_ROTATE);
    return k_rotate_attenuate(ctx, in, out, dims, axis, inv, delta, steps, z0, z_local);
}

// loop body S/SimulateMultiViewDataset.java:570-585 on device pointers
static int dev_simulate_view(mvsim_ctx* ctx, const mvsim_view_params* p, const float* gt, float* psf, float* out,
                             unsigned short* out16 = nullptr, int* d_overflow = nullptr)
{
    const size_t n = elems(p->dims);
    DevBufs bufs(ctx);
    float* a = bufs.alloc<float>(n);
    float* b = bufs.alloc<float>(n);
    MVSIM_TRY(bufs.st);
    // :570 + :573 in one pass (the rotated volume is not part of this entry point's output)
    const int st = dev_rotate_attenuate(ctx, gt, b, p->dims, p->axis, p->degrees, p->delta, p->strict_reference);
    if (st == MVSIM_EUNSUPPORTED) {
        MVSIM_TRY(dev_rotate(ctx, gt, a, p->dims, p->axis, p->degrees));
        MVSIM_TRY(dev_attenuate(ctx, a, b, p->dims, p->delta, p->strict_reference));
    } else if (st != MVSIM_OK) return st;
    // (Measured and dropped in round 2: the PSF chain -- normalise, x and y transforms, 0.26 ms -- on a side stream under
    // rotate_attenuate and the image's forward passes: 6.385 -> 6.345 ms per view with tools/time_view.py, but 6.2 -> 8.1 ms inside
    // bench.py's loop on a torch stream; the saturating main-stream kernels leave it nothing to hide behind.)
    MVSIM_TRY(dev_psf_normalize(ctx, psf, elems(p->kdims)));                                   // :255
    int planes = 0;
    MVSIM_TRY(conv_device(ctx, b, p->dims, psf, p->kdims, a, ctx->d_scalars + 1, p->inc, &planes));   // :580
    {
        StageTimer t(ctx, MVSIM_T_ADJUST);                                                     // :582, applied inside the sampler
        MVSIM_TRY(k_adjust_corr(ctx, ctx->d_scalars + 1, n, p->min_value, p->target_avg, ctx->d_scalars + 2));
    }
    StageTimer t(ctx, MVSIM_T_SAMPLE);                                                         // :585
    if (planes != p->dims[2]) {
        // the convolution already delivered the kept slices compacted (plus the sum plane, unused here)
        const int64_t kept[3] = { p->dims[0], p->dims[1], kept_planes(p->dims, p->inc) };
        return k_extract_u16(ctx, a, kept, 1, ctx->d_scalars + 2, p->min_value, p->snr, p->seed, p->stream, out, out16, d_overflow);
    }
    return k_extract_u16(ctx, a, p->dims, p->inc, ctx->d_scalars + 2, p->min_value, p->snr, p->seed, p->stream, out, out16, d_overflow);
}

// every view of a batch valid, all of them on the dims of the one ground truth (and of its resident volume, if there is one)
static int check_views(mvsim_ctx* ctx, int n, const mvsim_view_params* params, const mvsim_volume* vol, const char* what)
{
    for (int v = 0; v < n; ++v) {
        MVSIM_TRY(check_view(ctx, &params[v]));
        for (int d = 0; d < 3; ++d)
            if (params[v].dims[d] != params[0].dims[d] || (vol && vol->dims[d] != params[0].dims[d]))
                return set_error(ctx, MVSIM_EINVAL, "%s: all views share the ground truth dims", what);
    }
    return MVSIM_OK;
}

// Per-device phase gates of the batch calls: callers that run contexts concurrently on one GPU (the reference's tile
// stitching driver does, S/SimulateTileStitching.java:85-117) fall into a pipeline -- one uploads while the other computes.
struct DeviceGates { std::mutex upload, compute; };
static DeviceGates& gates_for(int device)
{
    static DeviceGates gates[64];
    return gates[(unsigned)device % 64];
}

// The protocol of the batch calls (DESIGN section 9): buffers and events first, then upload(), compute() and finish().  A
// failure is deferred: st keeps the first one, the later phases are skipped, and finish() still drains and frees, and returns it.
class BatchCall : public DevBufs {
public:
    BatchCall(mvsim_ctx* c, const char* what) : DevBufs(c), what_(what), gates_(gates_for(c->device))
    {
        stamp("enter");
        cudaError_t e = cudaSuccess;
        if (!ctx->copy_stream && (e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) {
            ctx->copy_stream = nullptr;
            st = cuda_fail(ctx, e, "cudaStreamCreateWithFlags");
        }
        mark_ = event();
    }
    ~BatchCall() { for (cudaEvent_t e : events_) cudaEventDestroy(e); }

    // an event of this call, destroyed with it; null after a failure
    cudaEvent_t event()
    {
        cudaEvent_t e = nullptr;
        if (st == MVSIM_OK && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess)
            st = set_error(ctx, MVSIM_ECUDA, "%s: cannot create events", what_);
        if (st != MVSIM_OK) return nullptr;
        events_.push_back(e);
        return e;
    }

    // the ground truth on the device: the resident volume, or a buffer that upload() fills from `host` before anything else
    const float* ground_truth(const float* host, const mvsim_volume* vol, size_t n)
    {
        if (vol) return vol->d;
        gt_host_ = host; gt_bytes_ = n * sizeof(float);
        return gt_dev_ = alloc<float>(n);
    }

    // Upload gate: two contexts never share the host->device link, so the second caller's upload runs at full rate under the
    // first caller's kernels instead of both uploads at half rate followed by both kernel phases.  ALL of a call's uploads
    // happen here (enqueue() issues those after the ground truth): a PSF upload issued later would queue on the copy engine
    // behind the other caller's 2 GB ground truth and stall this context's kernels for the length of that transfer.
    template <class Enqueue> void upload(Enqueue enqueue)
    {
        if (st != MVSIM_OK) return;
        {
            std::lock_guard<std::mutex> lk(gates_.upload);
            stamp("upload gate");
            if (gt_host_) st = h2d(ctx, gt_dev_, gt_host_, gt_bytes_);
            if (st == MVSIM_OK) st = enqueue();
            if (st == MVSIM_OK && (cudaEventRecord(mark_, ctx->stream) != cudaSuccess || cudaEventSynchronize(mark_) != cudaSuccess))
                st = set_error(ctx, MVSIM_ECUDA, "%s: upload failed", what_);
        }
        if (st == MVSIM_OK) stamp("upload done");
    }

    // Compute gate: body(&last) enqueues the kernels and downloads and names the event recorded after the last kernel.  The
    // gate opens when that event has completed; the tail of the downloads overlaps the next caller's kernels.
    template <class Body> void compute(Body body)
    {
        if (st != MVSIM_OK) return;
        std::lock_guard<std::mutex> lk(gates_.compute);
        stamp("compute gate");
        cudaEvent_t last = nullptr;
        st = body(&last);
        if (st == MVSIM_OK && last && cudaEventSynchronize(last) != cudaSuccess) st = set_error(ctx, MVSIM_ECUDA, "%s: kernels failed", what_);
        stamp("kernels done");
    }

    int finish()
    {
        // the main stream waits for the copy stream before the buffers go back to the pool
        if (mark_ && cudaEventRecord(mark_, ctx->copy_stream) == cudaSuccess) cudaStreamWaitEvent(ctx->stream, mark_, 0);
        free_all();
        const int st2 = sync(ctx);
        stamp("downloads done");
        return st != MVSIM_OK ? st : st2;
    }

    void stamp(const char* what) const
    {
        static const bool trace = getenv("MVSIM_TRACE") != nullptr;
        if (trace) fprintf(stderr, "[mvsim %p] %10.3f ms %s\n", (void*)ctx, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(), what);
    }

private:
    const char* what_;
    DeviceGates& gates_;
    std::vector<cudaEvent_t> events_;
    cudaEvent_t mark_ = nullptr;            // end of the uploads, then end of the copy stream's work
    const float* gt_host_ = nullptr;
    float* gt_dev_ = nullptr;
    size_t gt_bytes_ = 0;
};

}  // namespace mvsim

using namespace mvsim;

extern "C" {

int mvsim_version(void) { return 100; }

int mvsim_device_count(int* count)
{
    if (!count) return MVSIM_EINVAL;
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess) { *count = 0; return cuda_fail(nullptr, e, "cudaGetDeviceCount"); }
    return MVSIM_OK;
}

static int ctx_create(int device, bool own, void* cuda_stream, mvsim_ctx** out)
{
    if (!out) return set_error(nullptr, MVSIM_EINVAL, "null output pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n < 1)
        return set_error(nullptr, MVSIM_ECUDA, "no CUDA device available (%s); libmvsim has no CPU fallback",
                         e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return set_error(nullptr, MVSIM_EINVAL, "device %d out of range [0,%d)", device, n);
    DeviceScope scope(device);
    if (!scope.ok) return set_error(nullptr, MVSIM_ECUDA, "cannot select CUDA device %d", device);
    mvsim_ctx* ctx = new mvsim_ctx();
    ctx->device = device;
    ctx->stream = nullptr;
    ctx->own_stream = false;
    ctx->copy_stream = nullptr;
    ctx->mempool = nullptr;
    ctx->d_scalars = nullptr;
    ctx->launches = 0;
    ctx->psf_cache_max_bytes = 0;
    ctx->psf_cache_tick = ctx->psf_cache_hits = ctx->psf_cache_misses = 0;
    ctx->d_hash = nullptr;
    ctx->h_hash = nullptr;
    ctx->count_transport = 0;
    ctx->host_threads = 0;
    {
        // A/B runs without touching the caller: MVSIM_Z_KERNEL=<0..3> presets MVSIM_OPT_Z_KERNEL
        const char* zk = getenv("MVSIM_Z_KERNEL");
        const int v = zk ? atoi(zk) : 0;
        ctx->z_kernel = (v >= 0 && v <= 3) ? v : 0;
    }
    ctx->widen_pool = nullptr;
    ctx->profiling = false;
    memset(ctx->acc_ms, 0, sizeof(ctx->acc_ms));
    memset(ctx->acc_n, 0, sizeof(ctx->acc_n));
    int st = MVSIM_OK;
    do {
        if (!own) ctx->stream = static_cast<cudaStream_t>(cuda_stream);     // NULL = the legacy default stream
        else {
            if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) { st = cuda_fail(nullptr, e, "cudaStreamCreate"); break; }
            ctx->own_stream = true;
        }
        if ((e = cudaMalloc((void**)&ctx->d_scalars, 8 * sizeof(double))) != cudaSuccess) { st = cuda_fail(nullptr, e, "cudaMalloc"); break; }
        // freed workspaces stay cached in a stream-ordered pool owned by this context (no per-call cudaMalloc, and no
        // cross-stream reuse dependencies between contexts that run concurrently)
        cudaMemPoolProps props;
        memset(&props, 0, sizeof(props));
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        if ((e = cudaMemPoolCreate(&ctx->mempool, &props)) != cudaSuccess) { st = cuda_fail(nullptr, e, "cudaMemPoolCreate"); ctx->mempool = nullptr; break; }
        uint64_t keep = ~0ull;
        cudaMemPoolSetAttribute(ctx->mempool, cudaMemPoolAttrReleaseThreshold, &keep);
    } while (0);
    if (st != MVSIM_OK) {
        if (ctx->mempool) cudaMemPoolDestroy(ctx->mempool);
        if (ctx->d_scalars) cudaFree(ctx->d_scalars);
        if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
        delete ctx;
        return st;
    }
    *out = ctx;
    return MVSIM_OK;
}

int mvsim_ctx_create(int device, mvsim_ctx** out) { return ctx_create(device, true, nullptr, out); }
int mvsim_ctx_create_on_stream(int device, void* cuda_stream, mvsim_ctx** out) { return ctx_create(device, false, cuda_stream, out); }

int mvsim_ctx_destroy(mvsim_ctx* ctx)
{
    if (!ctx) return MVSIM_OK;
    DeviceScope scope(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto& kv : ctx->tables) cudaFree(kv.second.tw);
    for (auto& kv : ctx->dec_tables) cudaFree(kv.second);
    for (auto& e : ctx->psf_cache) cudaFree(e.p2);
    if (ctx->d_hash) cudaFree(ctx->d_hash);
    if (ctx->h_hash) cudaFreeHost(ctx->h_hash);
    for (auto& st : ctx->staging) if (st.p) cudaFreeHost(st.p);
    delete static_cast<mvsim::WidenPool*>(ctx->widen_pool);
    for (auto& ev : ctx->events) { cudaEventDestroy(ev.a); cudaEventDestroy(ev.b); }
    for (auto& ev : ctx->pool) { cudaEventDestroy(ev.a); cudaEventDestroy(ev.b); }
    cudaFree(ctx->d_scalars);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->mempool) cudaMemPoolDestroy(ctx->mempool);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return MVSIM_OK;
}

int mvsim_ctx_synchronize(mvsim_ctx* ctx)
{
    MVSIM_ENTER(ctx);
    return sync(ctx);
}

const char* mvsim_last_error(mvsim_ctx* ctx) { return ctx ? ctx->err.c_str() : tls_error.c_str(); }

int mvsim_profile_enable(mvsim_ctx* ctx, int on)
{
    if (!ctx) return MVSIM_EINVAL;
    ctx->profiling = on != 0;
    return MVSIM_OK;
}

static int drain_events(mvsim_ctx* ctx)
{
    MVSIM_TRY(sync(ctx));
    for (auto& ev : ctx->events) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ev.a, ev.b) == cudaSuccess) {
            ctx->acc_ms[ev.stage] += ms;
            ctx->acc_n[ev.stage] += 1;
        }
        ctx->pool.push_back(ev);
    }
    ctx->events.clear();
    return MVSIM_OK;
}

int mvsim_profile_reset(mvsim_ctx* ctx)
{
    MVSIM_ENTER(ctx);
    MVSIM_TRY(drain_events(ctx));
    memset(ctx->acc_ms, 0, sizeof(ctx->acc_ms));
    memset(ctx->acc_n, 0, sizeof(ctx->acc_n));
    return MVSIM_OK;
}

int mvsim_stage_times(mvsim_ctx* ctx, double ms[MVSIM_NSTAGES], int64_t launches[MVSIM_NSTAGES])
{
    MVSIM_ENTER(ctx);
    MVSIM_TRY(drain_events(ctx));
    for (int i = 0; i < MVSIM_NSTAGES; ++i) {
        if (ms) ms[i] = ctx->acc_ms[i];
        if (launches) launches[i] = ctx->acc_n[i];
    }
    return MVSIM_OK;
}

int64_t mvsim_kernel_launches(mvsim_ctx* ctx) { return ctx ? ctx->launches : 0; }

int mvsim_ctx_set_option(mvsim_ctx* ctx, int option, int64_t value)
{
    if (!ctx) return set_error(nullptr, MVSIM_EINVAL, "null context");
    switch (option) {
    case MVSIM_OPT_COUNT_TRANSPORT:
        if (value != 0 && value != 1) return set_error(ctx, MVSIM_EINVAL, "count transport: 0 (float32) or 1 (uint16)");
        ctx->count_transport = (int)value;
        return MVSIM_OK;
    case MVSIM_OPT_HOST_THREADS:
        if (value < 0 || value > 256) return set_error(ctx, MVSIM_EINVAL, "host threads: 0 (default) .. 256");
        if (ctx->widen_pool) { delete static_cast<mvsim::WidenPool*>(ctx->widen_pool); ctx->widen_pool = nullptr; }
        ctx->host_threads = (int)value;
        return MVSIM_OK;
    case MVSIM_OPT_Z_KERNEL:
        if (value < 0 || value > 3) return set_error(ctx, MVSIM_EINVAL, "z kernel: 0 (auto), 1 (no polyphase), 2 (full spectral), 3 (polyphase)");
        ctx->z_kernel = (int)value;
        return MVSIM_OK;
    }
    return set_error(ctx, MVSIM_EINVAL, "unknown option %d", option);
}

int mvsim_psf_cache_configure(mvsim_ctx* ctx, size_t max_bytes)
{
    MVSIM_ENTER(ctx);
    MVSIM_TRY(sync(ctx));                       // nothing in flight reads an entry that is about to go
    if (max_bytes < ctx->psf_cache_max_bytes) {
        for (auto& e : ctx->psf_cache) cudaFree(e.p2);
        ctx->psf_cache.clear();
    }
    ctx->psf_cache_max_bytes = max_bytes;
    return MVSIM_OK;
}

int mvsim_psf_cache_stats(mvsim_ctx* ctx, int64_t stats[4])
{
    if (!ctx || !stats) return MVSIM_EINVAL;
    size_t held = 0;
    for (auto& e : ctx->psf_cache) held += e.bytes;
    stats[0] = (int64_t)ctx->psf_cache_hits; stats[1] = (int64_t)ctx->psf_cache_misses;
    stats[2] = (int64_t)ctx->psf_cache.size(); stats[3] = (int64_t)held;
    return MVSIM_OK;
}

int mvsim_alloc_pinned(size_t bytes, void** ptr)
{
    if (!ptr) return MVSIM_EINVAL;
    cudaError_t e = cudaHostAlloc(ptr, bytes ? bytes : 16, cudaHostAllocPortable);
    if (e != cudaSuccess) { *ptr = nullptr; return cuda_fail(nullptr, e, "cudaHostAlloc"); }
    return MVSIM_OK;
}

int mvsim_free_pinned(void* ptr)
{
    if (!ptr) return MVSIM_OK;
    cudaError_t e = cudaFreeHost(ptr);
    return e == cudaSuccess ? MVSIM_OK : cuda_fail(nullptr, e, "cudaFreeHost");
}

int mvsim_conv_padded_dims(const int64_t dims[3], const int64_t kdims[3], int64_t nfft[3])
{
    if (!dims || !kdims || !nfft) return MVSIM_EINVAL;
    ConvPlan pl;
    const int e = make_conv_plan(dims, kdims, &pl);
    if (e) return e == 1 ? MVSIM_EINVAL : MVSIM_EUNSUPPORTED;
    nfft[0] = 2 * pl.sx.n; nfft[1] = pl.sy.n; nfft[2] = pl.sz.n;
    return MVSIM_OK;
}

int mvsim_axis_rotation(const int64_t dims[3], int axis, int degrees, double fwd[12], double inv[12])
{
    if (!dims) return MVSIM_EINVAL;
    return axis_rotation(dims, axis, degrees, fwd, inv);
}

// ---- host-buffer entry points ---------------------------------------------------------------
int mvsim_rotate_axis(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], int axis, int degrees)
{
    MVSIM_ENTER(ctx);
    if (!in || !out) return set_error(ctx, MVSIM_EINVAL, "rotate: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "rotate"));
    HostCall hc(ctx);
    const float* a = hc.in(in, elems(dims));
    float* b = hc.out(out, elems(dims));
    return hc.run([&] { return dev_rotate(ctx, a, b, dims, axis, degrees); });
}

int mvsim_attenuate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], double delta, int strict_reference)
{
    MVSIM_ENTER(ctx);
    if (!in || !out) return set_error(ctx, MVSIM_EINVAL, "attenuate: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "attenuate"));
    HostCall hc(ctx);
    const float* a = hc.in(in, elems(dims));
    float* b = hc.out(out, elems(dims));
    return hc.run([&] { return dev_attenuate(ctx, a, b, dims, delta, strict_reference); });
}

int mvsim_psf_normalize(mvsim_ctx* ctx, float* psf, const int64_t kdims[3], double* sum_out)
{
    MVSIM_ENTER(ctx);
    if (!psf) return set_error(ctx, MVSIM_EINVAL, "psf_normalize: null buffer");
    MVSIM_TRY(check_dims(ctx, kdims, "psf_normalize"));
    HostCall hc(ctx);
    float* a = hc.inout(psf, elems(kdims));
    hc.scalar(0, sum_out);
    return hc.run([&] { return dev_psf_normalize(ctx, a, elems(kdims)); });
}

int mvsim_convolve(mvsim_ctx* ctx, const float* img, const int64_t dims[3], float* psf, const int64_t kdims[3], float* out)
{
    MVSIM_ENTER(ctx);
    if (!img || !psf || !out) return set_error(ctx, MVSIM_EINVAL, "convolve: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "convolve dims"));
    MVSIM_TRY(check_dims(ctx, kdims, "convolve kdims"));
    HostCall hc(ctx);
    const float* a = hc.in(img, elems(dims));
    float* b = hc.out(out, elems(dims));
    float* k = hc.inout(psf, elems(kdims));          // in-place normalisation is part of the contract (:255)
    return hc.run([&] {
        MVSIM_TRY(dev_psf_normalize(ctx, k, elems(kdims)));
        return conv_device(ctx, a, dims, k, kdims, b, nullptr);
    });
}

int mvsim_adjust(mvsim_ctx* ctx, float* img, const int64_t dims[3], float min_value, float target_avg, double* correction_out)
{
    MVSIM_ENTER(ctx);
    if (!img) return set_error(ctx, MVSIM_EINVAL, "adjust: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "adjust"));
    HostCall hc(ctx);
    float* a = hc.inout(img, elems(dims));
    hc.scalar(2, correction_out);
    return hc.run([&] { return dev_adjust(ctx, a, elems(dims), min_value, target_avg); });
}

int mvsim_extract_slices(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, float snr, uint64_t seed, uint64_t stream, float* out)
{
    MVSIM_ENTER(ctx);
    if (!in || !out) return set_error(ctx, MVSIM_EINVAL, "extract_slices: null buffer");
    MVSIM_TRY(check_sampling(ctx, dims, inc, "extract_slices"));
    HostCall hc(ctx);
    const float* a = hc.in(in, elems(dims));
    float* b = hc.out(out, kept_elems(dims, inc));
    return hc.run([&] { return dev_extract_slices(ctx, a, dims, inc, snr, seed, stream, b); });
}

int mvsim_poisson(mvsim_ctx* ctx, float* inout, size_t n, double snr, uint64_t seed, uint64_t stream)
{
    MVSIM_ENTER(ctx);
    if (!inout && n) return set_error(ctx, MVSIM_EINVAL, "poisson: null buffer");
    if (n == 0) return MVSIM_OK;
    HostCall hc(ctx);
    float* a = hc.inout(inout, n);
    return hc.run([&] {
        StageTimer t(ctx, MVSIM_T_SAMPLE);
        return k_poisson(ctx, a, n, snr, seed, stream);
    });
}

int mvsim_simulate_view(mvsim_ctx* ctx, const mvsim_view_params* p, const float* gt, float* psf, float* out)
{
    MVSIM_ENTER(ctx);
    MVSIM_TRY(check_view(ctx, p));
    if (!gt || !psf || !out) return set_error(ctx, MVSIM_EINVAL, "simulate_view: null buffer");
    HostCall hc(ctx);
    const float* g = hc.in(gt, elems(p->dims));
    float* k = hc.inout(psf, elems(p->kdims));
    float* o = hc.out(out, kept_elems(p->dims, p->inc));
    return hc.run([&] { return dev_simulate_view(ctx, p, g, k, o); });
}

// gt: host ground truth (uploaded under the upload gate) or, when vol is given, already resident on the device
static int simulate_views_impl(mvsim_ctx* ctx, int n_views, const mvsim_view_params* params, const float* gt, const mvsim_volume* vol,
                               float* const* psfs, float* const* outs)
{
    if (n_views < 0 || (n_views > 0 && (!params || (!gt && !vol) || !psfs || !outs))) return set_error(ctx, MVSIM_EINVAL, "simulate_views: null argument");
    if (n_views == 0) return MVSIM_OK;
    MVSIM_TRY(check_views(ctx, n_views, params, vol, "simulate_views"));
    for (int v = 0; v < n_views; ++v)
        if (!psfs[v] || !outs[v]) return set_error(ctx, MVSIM_EINVAL, "simulate_views: null buffer for view %d", v);
    BatchCall bc(ctx, "simulate_views");
    const float* gt_dev = bc.ground_truth(gt, vol, elems(params[0].dims));
    cudaEvent_t done = bc.event();
    // every view's device PSF and output stay alive until its download is done
    std::vector<float*> k((size_t)n_views), o((size_t)n_views);
    for (int v = 0; v < n_views; ++v) {
        k[(size_t)v] = bc.alloc<float>(elems(params[v].kdims));
        o[(size_t)v] = bc.alloc<float>(kept_elems(params[v].dims, params[v].inc));
    }
    // Count transport (MVSIM_OPT_COUNT_TRANSPORT, views with Poisson noise): the sampler also writes the counts as uint16; those
    // cross the link into a pinned staging buffer and host threads widen them into the caller's float32 buffer while later views
    // still compute / copy.  A view whose counts exceed 65535 (flag) is fetched again as float32.
    struct U16View { unsigned short* d16; unsigned short* h16; int* d_flag; int* h_flag; cudaEvent_t copied; bool on; };
    std::vector<U16View> u16((size_t)n_views, U16View{ nullptr, nullptr, nullptr, nullptr, nullptr, false });
    if (bc.st == MVSIM_OK && ctx->count_transport == 1) {
        void* h_flags = nullptr;
        bc.st = staging_buffer(ctx, 0, (size_t)n_views * sizeof(int) + 64, &h_flags);
        for (int v = 0; v < n_views && bc.st == MVSIM_OK; ++v) {
            if (!(params[v].snr >= 0.0f)) continue;
            const size_t n_out = kept_elems(params[v].dims, params[v].inc);
            U16View& u = u16[(size_t)v];
            u.d16 = bc.alloc<unsigned short>(n_out);
            u.d_flag = bc.alloc<int>(4);
            void* h16 = nullptr;
            if (bc.st == MVSIM_OK) bc.st = staging_buffer(ctx, (size_t)v + 1, n_out * sizeof(unsigned short), &h16);
            u.h16 = static_cast<unsigned short*>(h16);
            u.h_flag = static_cast<int*>(h_flags) + v;
            u.copied = bc.event();
            u.on = bc.st == MVSIM_OK;
        }
    }
    int next_u16 = 0;
    auto finish_u16 = [&](int v) -> int {
        U16View& u = u16[(size_t)v];
        if (!u.on) return MVSIM_OK;
        if (cudaEventSynchronize(u.copied) != cudaSuccess) return set_error(ctx, MVSIM_ECUDA, "simulate_views: download failed");
        const size_t n_out = kept_elems(params[v].dims, params[v].inc);
        if (*u.h_flag) {
            // counts beyond uint16: this view travels as float32 after all
            cudaError_t e = cudaMemcpyAsync(outs[v], o[(size_t)v], n_out * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->copy_stream);
            if (e != cudaSuccess) return cuda_fail(ctx, e, "simulate_views: float32 fallback download");
        } else {
            const auto t0 = std::chrono::steady_clock::now();
            widen_pool(ctx)->run(u.h16, outs[v], n_out);
            if (ctx->profiling) {
                ctx->acc_ms[MVSIM_T_WIDEN] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
                ctx->acc_n[MVSIM_T_WIDEN] += 1;
            }
        }
        return MVSIM_OK;
    };
    bc.upload([&]() -> int {
        int st = MVSIM_OK;
        for (int v = 0; v < n_views && st == MVSIM_OK; ++v) st = h2d(ctx, k[(size_t)v], psfs[v], elems(params[v].kdims) * sizeof(float));
        return st;
    });
    bc.compute([&](cudaEvent_t* last) -> int {
        int st = MVSIM_OK;
        for (int v = 0; v < n_views && st == MVSIM_OK; ++v) {
            const mvsim_view_params* p = &params[v];
            const size_t n_out = kept_elems(p->dims, p->inc);
            U16View& u = u16[(size_t)v];
            cudaError_t e = cudaSuccess;
            if (u.on) e = cudaMemsetAsync(u.d_flag, 0, sizeof(int), ctx->stream);
            if (e != cudaSuccess) { st = cuda_fail(ctx, e, "simulate_views: flag"); break; }
            if ((st = dev_simulate_view(ctx, p, gt_dev, k[(size_t)v], o[(size_t)v], u.on ? u.d16 : nullptr, u.on ? u.d_flag : nullptr)) != MVSIM_OK) break;
            e = cudaEventRecord(done, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, done, 0);
            if (e == cudaSuccess) e = cudaMemcpyAsync(psfs[v], k[(size_t)v], elems(p->kdims) * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_stream);
            if (u.on) {
                if (e == cudaSuccess) e = cudaMemcpyAsync(u.h_flag, u.d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->copy_stream);
                if (e == cudaSuccess) e = cudaMemcpyAsync(u.h16, u.d16, n_out * sizeof(unsigned short), cudaMemcpyDeviceToHost, ctx->copy_stream);
                if (e == cudaSuccess) e = cudaEventRecord(u.copied, ctx->copy_stream);
            } else if (e == cudaSuccess) {
                e = cudaMemcpyAsync(outs[v], o[(size_t)v], n_out * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_stream);
            }
            if (e != cudaSuccess) st = cuda_fail(ctx, e, "simulate_views: download");
        }
        bc.stamp("enqueued");
        // uint16 views: as each copy lands, widen it into the caller's buffer while the later views still compute / copy -- but
        // only until this call's last kernel has run: then the gate opens and the rest is finished outside it
        while (st == MVSIM_OK && next_u16 < n_views - 1 && cudaEventQuery(done) == cudaErrorNotReady) st = finish_u16(next_u16++);
        cudaGetLastError();     // cudaErrorNotReady from the query is not an error
        *last = done;
        return st;
    });
    while (bc.st == MVSIM_OK && next_u16 < n_views) bc.st = finish_u16(next_u16++);
    return bc.finish();
}

int mvsim_simulate_views(mvsim_ctx* ctx, int n_views, const mvsim_view_params* params, const float* gt,
                         float* const* psfs, float* const* outs)
{
    MVSIM_ENTER(ctx);
    return simulate_views_impl(ctx, n_views, params, gt, nullptr, psfs, outs);
}

int mvsim_dev_simulate_views(mvsim_ctx* ctx, int n_views, const mvsim_view_params* params, const mvsim_volume* gt,
                             float* const* psfs, float* const* outs)
{
    MVSIM_ENTER(ctx);
    return simulate_views_impl(ctx, n_views, params, nullptr, gt, psfs, outs);
}

// ---- post-acquisition chain ---------------------------------------------------------------------
int mvsim_make_isotropic(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, float* out)
{
    MVSIM_ENTER(ctx);
    if (!in || !out) return set_error(ctx, MVSIM_EINVAL, "make_isotropic: null buffer");
    MVSIM_TRY(check_sampling(ctx, dims, inc, "make_isotropic"));
    HostCall hc(ctx);
    const float* a = hc.in(in, elems(dims));
    float* b = hc.out(out, (size_t)(dims[0] * dims[1] * ((dims[2] - 1) * inc + 1)));
    return hc.run([&] { return k_make_isotropic(ctx, a, dims, inc, b); });
}

int mvsim_weight_image(mvsim_ctx* ctx, const int64_t dims[3], float* out)
{
    MVSIM_ENTER(ctx);
    if (!out) return set_error(ctx, MVSIM_EINVAL, "weight_image: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "weight_image"));
    HostCall hc(ctx);
    float* a = hc.out(out, elems(dims));
    return hc.run([&] { return k_weight_image(ctx, dims, a); });
}

int mvsim_normalize_weights(mvsim_ctx* ctx, float* const* weights, int n_views, const int64_t dims[3], float osem, float* sum_out)
{
    MVSIM_ENTER(ctx);
    if (!weights || n_views < 1 || n_views > MVSIM_MAX_WEIGHT_VIEWS) return set_error(ctx, MVSIM_EINVAL, "normalize_weights: 1..%d views", MVSIM_MAX_WEIGHT_VIEWS);
    MVSIM_TRY(check_dims(ctx, dims, "normalize_weights"));
    for (int v = 0; v < n_views; ++v)
        if (!weights[v]) return set_error(ctx, MVSIM_EINVAL, "normalize_weights: null buffer");
    HostCall hc(ctx);
    float* d[MVSIM_MAX_WEIGHT_VIEWS] = {};
    for (int v = 0; v < n_views; ++v) d[v] = hc.inout(weights[v], elems(dims));
    float* dsum = sum_out ? hc.out(sum_out, elems(dims)) : nullptr;
    return hc.run([&] { return k_normalize_weights(ctx, d, n_views, elems(dims), osem, dsum); });
}

// ---- input generators either side of the path (SURVEY section 8f rows 2-4) -------------------------
namespace mvsim {
// java.util.Random (JDK specification): 48-bit LCG.  The reference draws bead positions (S/SimulateBeads.java:69,150-166)
// and the sphere phantom (S/SimulateMultiViewDataset.java:76,485,506,512) from it; replaying it keeps the caller's seeds.
struct JavaRandom {
    uint64_t s;
    explicit JavaRandom(int64_t seed) : s(((uint64_t)seed ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1)) {}
    int32_t next(int bits)
    {
        s = (s * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
        return (int32_t)(int64_t)(s >> (48 - bits));
    }
    double next_double() { const int64_t a = next(26), b = next(27); return (double)((a << 27) + b) * 0x1.0p-53; }
    int32_t next_int(int32_t bound)
    {
        int32_t r = next(31);
        const int32_t m = bound - 1;
        if ((bound & m) == 0) return (int32_t)(((int64_t)bound * (int64_t)r) >> 31);
        for (int32_t u = r; (int32_t)((uint32_t)u - (uint32_t)(r = u % bound) + (uint32_t)m) < 0; u = next(31)) {}
        return r;
    }
};

// drawSpheres (:436-522): walk the large sphere in HyperSphereCursor order (z, y, x ascending, nested integer radii),
// two draws per voxel, a third for the one voxel in ~2900 that gets a small sphere.  Only this replay is sequential.
static void replay_draw_spheres(const int64_t dims[3], double minv, double maxv, int scale, int half_pixel, int64_t seed,
                                std::vector<int>& rec, std::vector<float>& val)
{
    JavaRandom rnd(seed);
    int64_t c[3], min_size = dims[0];
    for (int d = 0; d < 3; ++d) { c[d] = dims[d] / 2; min_size = dims[d] < min_size ? dims[d] : min_size; }
    const int64_t R = min_size / 2 - 47 * scale - 1;                                         // :462
    const int max_radius = 10 * scale;                                                        // :458
    const int64_t mod = (int64_t)(7 * scale) * (7 * scale) * (7 * scale);                     // Util.pow(7*scale, 3), :509
    for (int64_t dz = -R; dz <= R; ++dz) {
        const int64_t ry = (int64_t)sqrt((double)(R * R - dz * dz));
        for (int64_t dy = -ry; dy <= ry; ++dy) {
            const int64_t rx = (int64_t)sqrt((double)(ry * ry - dy * dy));
            for (int64_t dx = -rx; dx <= rx; ++dx) {
                const int radius = rnd.next_int(max_radius) + 1;                              // :485
                const double rv = rnd.next_double();                                          // :506
                if ((int64_t)floor(rv * 10000 + 0.5) % mod != 0) continue;                    // Math.round, :509
                const double v = rnd.next_double() * (maxv - minv) + minv;                    // :512
                const int shift = half_pixel ? 1 : 0;                                         // :496-499, all but the last dimension
                rec.push_back((int)(c[0] + dx + shift));
                rec.push_back((int)(c[1] + dy + shift));
                rec.push_back((int)(c[2] + dz));
                rec.push_back(radius);
                val.push_back((float)v);
            }
        }
    }
}

static int dev_draw_spheres(mvsim_ctx* ctx, const int64_t dims[3], double minv, double maxv, int scale, int half_pixel, int64_t seed,
                            float* d_out, int64_t* n_small)
{
    if (scale < 1 || scale > 64) return set_error(ctx, MVSIM_EINVAL, "draw_spheres: scale must be in 1..64");
    if (!(minv >= 0.0) || !(maxv >= minv)) return set_error(ctx, MVSIM_EINVAL, "draw_spheres: need 0 <= minValue <= maxValue");
    std::vector<int> rec;
    std::vector<float> val;
    replay_draw_spheres(dims, minv, maxv, scale, half_pixel, seed, rec, val);
    if (n_small) *n_small = (int64_t)val.size();
    return k_paint_spheres(ctx, d_out, dims, rec.data(), val.data(), (int)val.size());
}

// simulate(halfPixelOffset, rnd) (:371-392): (size+1)*2 cube rendered, then downSample2x -> size^3
static int dev_simulate_phantom(mvsim_ctx* ctx, int size, int half_pixel, int64_t seed, float* d_out, int64_t* n_small)
{
    const int scale = 2;
    const int64_t big = (int64_t)(size + 1) * scale;
    const int64_t dims[3] = { big, big, big };
    DevBufs bufs(ctx);
    float* a = bufs.alloc<float>((size_t)(big * big * big));
    MVSIM_TRY(bufs.st);
    MVSIM_TRY(dev_draw_spheres(ctx, dims, 0.0, 1.0, scale, half_pixel, seed, a, n_small));
    return k_downsample2x(ctx, a, dims, d_out);
}

static int check_phantom_size(mvsim_ctx* ctx, int size)
{
    if (size < 1 || size > 2047) return set_error(ctx, MVSIM_EINVAL, "simulate_phantom: size must be in 1..2047");
    return MVSIM_OK;
}
}  // namespace mvsim
using namespace mvsim;

int mvsim_random_points(int n, const int64_t range_min[3], const int64_t range_max[3], int64_t seed, double* points)
{
    if (n < 0 || !range_min || !range_max || (n > 0 && !points)) return set_error(nullptr, MVSIM_EINVAL, "random_points: bad argument");
    JavaRandom rnd(seed);
    for (int i = 0; i < n; ++i)
        for (int d = 0; d < 3; ++d)
            points[3 * i + d] = rnd.next_double() * (double)(range_max[d] - range_min[d]) + (double)range_min[d];     // :161
    return MVSIM_OK;
}

int mvsim_transform_points(const double* points, int n, const int64_t range_min[3], const int64_t range_max[3], int axis, int degrees, double* out)
{
    if (n < 0 || !range_min || !range_max || (n > 0 && (!points || !out))) return set_error(nullptr, MVSIM_EINVAL, "transform_points: bad argument");
    int64_t dims[3];
    for (int d = 0; d < 3; ++d) dims[d] = range_max[d] - range_min[d] + 1;          // axisRotation uses (max - min) / 2
    double m[12];
    if (axis_rotation(dims, axis, degrees, m, nullptr)) return set_error(nullptr, MVSIM_EINVAL, "transform_points: axis must be 0, 1 or 2");
    for (int i = 0; i < n; ++i) {
        const double p0 = points[3 * i], p1 = points[3 * i + 1], p2 = points[3 * i + 2];
        for (int r = 0; r < 3; ++r) out[3 * i + r] = p0 * m[4 * r] + p1 * m[4 * r + 1] + p2 * m[4 * r + 2] + m[4 * r + 3];
    }
    return MVSIM_OK;
}

static int check_bead_args(mvsim_ctx* ctx, const double* points, int n, const double sigma[3], const int64_t imin[3], const int64_t imax[3], int64_t dims[3])
{
    if (n < 0 || (n > 0 && !points) || !sigma || !imin || !imax) return set_error(ctx, MVSIM_EINVAL, "render_beads: null argument");
    for (int d = 0; d < 3; ++d) {
        if (!(sigma[d] > 0) || sigma[d] > 1000) return set_error(ctx, MVSIM_EINVAL, "render_beads: sigma must be in (0, 1000]");
        dims[d] = imax[d] - imin[d];
    }
    return check_dims(ctx, dims, "render_beads (image dims = max - min)");
}

int mvsim_render_beads(mvsim_ctx* ctx, const double* points, int n, const double sigma[3], const int64_t imin[3], const int64_t imax[3], float* out)
{
    MVSIM_ENTER(ctx);
    int64_t dims[3];
    MVSIM_TRY(check_bead_args(ctx, points, n, sigma, imin, imax, dims));
    if (!out) return set_error(ctx, MVSIM_EINVAL, "render_beads: null buffer");
    HostCall hc(ctx);
    float* a = hc.out(out, elems(dims));
    return hc.run([&] { return k_render_beads(ctx, points, n, sigma, imin, imax, a); });
}

int mvsim_dev_render_beads(mvsim_ctx* ctx, const double* points, int n, const double sigma[3], const int64_t imin[3], const int64_t imax[3], mvsim_volume* out)
{
    MVSIM_ENTER(ctx);
    int64_t dims[3];
    MVSIM_TRY(check_bead_args(ctx, points, n, sigma, imin, imax, dims));
    if (!out || out->dims[0] != dims[0] || out->dims[1] != dims[1] || out->dims[2] != dims[2])
        return set_error(ctx, MVSIM_EINVAL, "render_beads: output volume must have dims max - min");
    return k_render_beads(ctx, points, n, sigma, imin, imax, out->d);
}

int mvsim_draw_spheres(mvsim_ctx* ctx, const int64_t dims[3], double min_value, double max_value, int scale, int half_pixel, int64_t seed,
                       float* out, int64_t* n_small)
{
    MVSIM_ENTER(ctx);
    if (!out) return set_error(ctx, MVSIM_EINVAL, "draw_spheres: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "draw_spheres"));
    HostCall hc(ctx);
    float* a = hc.out(out, elems(dims));
    return hc.run([&] { return dev_draw_spheres(ctx, dims, min_value, max_value, scale, half_pixel, seed, a, n_small); });
}

int mvsim_downsample2x(mvsim_ctx* ctx, const float* in, const int64_t dims[3], float* out)
{
    MVSIM_ENTER(ctx);
    if (!in || !out) return set_error(ctx, MVSIM_EINVAL, "downsample2x: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "downsample2x"));
    if (dims[0] < 4 || dims[1] < 4 || dims[2] < 4) return set_error(ctx, MVSIM_EINVAL, "downsample2x: dims must be >= 4 (output is dims/2 - 1)");
    HostCall hc(ctx);
    const float* a = hc.in(in, elems(dims));
    float* b = hc.out(out, (size_t)((dims[0] / 2 - 1) * (dims[1] / 2 - 1) * (dims[2] / 2 - 1)));
    return hc.run([&] { return k_downsample2x(ctx, a, dims, b); });
}

int mvsim_simulate_phantom(mvsim_ctx* ctx, int size, int half_pixel, int64_t seed, float* out, int64_t* n_small)
{
    MVSIM_ENTER(ctx);
    if (!out) return set_error(ctx, MVSIM_EINVAL, "simulate_phantom: null buffer");
    MVSIM_TRY(check_phantom_size(ctx, size));
    HostCall hc(ctx);
    float* b = hc.out(out, (size_t)size * size * size);
    return hc.run([&] { return dev_simulate_phantom(ctx, size, half_pixel, seed, b, n_small); });
}

int mvsim_dev_simulate_phantom(mvsim_ctx* ctx, int size, int half_pixel, int64_t seed, mvsim_volume* out, int64_t* n_small)
{
    MVSIM_ENTER(ctx);
    MVSIM_TRY(check_phantom_size(ctx, size));
    if (!out || out->dims[0] != size || out->dims[1] != size || out->dims[2] != size)
        return set_error(ctx, MVSIM_EINVAL, "simulate_phantom: output volume must be size^3");
    return dev_simulate_phantom(ctx, size, half_pixel, seed, out->d, n_small);
}

int mvsim_make_square(mvsim_ctx* ctx, const float* in, const int64_t dims[3], float* out)
{
    MVSIM_ENTER(ctx);
    if (!in || !out) return set_error(ctx, MVSIM_EINVAL, "make_square: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "make_square"));
    const int64_t m = dims[0] > dims[1] ? (dims[0] > dims[2] ? dims[0] : dims[2]) : (dims[1] > dims[2] ? dims[1] : dims[2]);
    if (m > 4096) return set_error(ctx, MVSIM_EINVAL, "make_square: dims too large");
    HostCall hc(ctx);
    const float* a = hc.in(in, elems(dims));
    float* b = hc.out(out, (size_t)(m * m * m));
    return hc.run([&] { return k_make_square(ctx, a, dims, b); });
}

// ---- device-resident volumes ------------------------------------------------------------------
int mvsim_volume_create(mvsim_ctx* ctx, const int64_t dims[3], mvsim_volume** vol)
{
    MVSIM_ENTER(ctx);
    if (!vol) return set_error(ctx, MVSIM_EINVAL, "volume_create: null output pointer");
    *vol = nullptr;
    MVSIM_TRY(check_dims(ctx, dims, "volume_create"));
    mvsim_volume* v = new mvsim_volume();
    v->device = ctx->device;
    memcpy(v->dims, dims, sizeof(v->dims));
    cudaError_t e = cudaMalloc((void**)&v->d, v->elems() * sizeof(float));
    if (e != cudaSuccess) { delete v; return cuda_fail(ctx, e, "cudaMalloc(volume)"); }
    *vol = v;
    return MVSIM_OK;
}

int mvsim_volume_wrap(mvsim_ctx* ctx, const int64_t dims[3], void* device_ptr, mvsim_volume** vol)
{
    MVSIM_ENTER(ctx);
    if (!vol || !device_ptr) return set_error(ctx, MVSIM_EINVAL, "volume_wrap: null argument");
    *vol = nullptr;
    MVSIM_TRY(check_dims(ctx, dims, "volume_wrap"));
    if (reinterpret_cast<uintptr_t>(device_ptr) % 16) return set_error(ctx, MVSIM_EINVAL, "volume_wrap: device pointer must be 16-byte aligned");
    mvsim_volume* v = new mvsim_volume();
    v->device = ctx->device;
    memcpy(v->dims, dims, sizeof(v->dims));
    v->d = static_cast<float*>(device_ptr);
    v->borrowed = true;
    *vol = v;
    return MVSIM_OK;
}

int mvsim_volume_free(mvsim_ctx* ctx, mvsim_volume* vol)
{
    if (!vol) return MVSIM_OK;
    MVSIM_ENTER(ctx);
    cudaStreamSynchronize(ctx->stream);
    if (!vol->borrowed) cudaFree(vol->d);
    delete vol;
    return MVSIM_OK;
}

int mvsim_volume_dims(const mvsim_volume* vol, int64_t dims[3])
{
    if (!vol || !dims) return MVSIM_EINVAL;
    memcpy(dims, vol->dims, sizeof(vol->dims));
    return MVSIM_OK;
}

void* mvsim_volume_device_ptr(mvsim_volume* vol) { return vol ? vol->d : nullptr; }

int mvsim_volume_upload(mvsim_ctx* ctx, mvsim_volume* vol, const float* host)
{
    MVSIM_ENTER(ctx);
    if (!vol || !host) return set_error(ctx, MVSIM_EINVAL, "volume_upload: null argument");
    return h2d(ctx, vol->d, host, vol->elems() * sizeof(float));
}

int mvsim_volume_download(mvsim_ctx* ctx, const mvsim_volume* vol, float* host)
{
    MVSIM_ENTER(ctx);
    if (!vol || !host) return set_error(ctx, MVSIM_EINVAL, "volume_download: null argument");
    return d2h(ctx, host, vol->d, vol->elems() * sizeof(float));
}

static bool same_dims(const mvsim_volume* a, const mvsim_volume* b)
{
    return a->dims[0] == b->dims[0] && a->dims[1] == b->dims[1] && a->dims[2] == b->dims[2];
}

int mvsim_dev_rotate_axis(mvsim_ctx* ctx, const mvsim_volume* in, mvsim_volume* out, int axis, int degrees)
{
    MVSIM_ENTER(ctx);
    if (!in || !out || in == out || !same_dims(in, out)) return set_error(ctx, MVSIM_EINVAL, "dev_rotate: need two distinct volumes of equal dims");
    return dev_rotate(ctx, in->d, out->d, in->dims, axis, degrees);
}

int mvsim_dev_attenuate(mvsim_ctx* ctx, const mvsim_volume* in, mvsim_volume* out, double delta, int strict_reference)
{
    MVSIM_ENTER(ctx);
    if (!in || !out || in == out || !same_dims(in, out)) return set_error(ctx, MVSIM_EINVAL, "dev_attenuate: need two distinct volumes of equal dims");
    return dev_attenuate(ctx, in->d, out->d, in->dims, delta, strict_reference);
}

int mvsim_dev_psf_normalize(mvsim_ctx* ctx, mvsim_volume* psf, double* sum_out)
{
    MVSIM_ENTER(ctx);
    if (!psf) return set_error(ctx, MVSIM_EINVAL, "dev_psf_normalize: null volume");
    MVSIM_TRY(dev_psf_normalize(ctx, psf->d, psf->elems()));
    if (sum_out) MVSIM_TRY(read_scalar(ctx, 0, sum_out));
    return MVSIM_OK;
}

int mvsim_dev_convolve(mvsim_ctx* ctx, const mvsim_volume* img, const mvsim_volume* psf, mvsim_volume* out)
{
    MVSIM_ENTER(ctx);
    if (!img || !psf || !out || img == out || !same_dims(img, out)) return set_error(ctx, MVSIM_EINVAL, "dev_convolve: need img/out of equal dims, distinct");
    return conv_device(ctx, img->d, img->dims, psf->d, psf->dims, out->d, nullptr);
}

int mvsim_dev_adjust(mvsim_ctx* ctx, mvsim_volume* img, float min_value, float target_avg, double* correction_out)
{
    MVSIM_ENTER(ctx);
    if (!img) return set_error(ctx, MVSIM_EINVAL, "dev_adjust: null volume");
    MVSIM_TRY(dev_adjust(ctx, img->d, img->elems(), min_value, target_avg));
    if (correction_out) MVSIM_TRY(read_scalar(ctx, 2, correction_out));
    return MVSIM_OK;
}

int mvsim_dev_extract_slices(mvsim_ctx* ctx, const mvsim_volume* in, int inc, float snr, uint64_t seed, uint64_t stream, mvsim_volume* out)
{
    MVSIM_ENTER(ctx);
    if (!in || !out) return set_error(ctx, MVSIM_EINVAL, "dev_extract_slices: null volume");
    MVSIM_TRY(check_sampling(ctx, in->dims, inc, "dev_extract_slices"));
    if (out->dims[0] != in->dims[0] || out->dims[1] != in->dims[1] || out->dims[2] != kept_planes(in->dims, inc))
        return set_error(ctx, MVSIM_EINVAL, "dev_extract_slices: out dims must be (X, Y, (Z-1)/inc+1)");
    return dev_extract_slices(ctx, in->d, in->dims, inc, snr, seed, stream, out->d);
}

int mvsim_dev_extract_interval(mvsim_ctx* ctx, const mvsim_volume* in, const int64_t min[3], const int64_t max[3], int inc,
                               float snr, uint64_t seed, uint64_t stream, mvsim_volume* out)
{
    MVSIM_ENTER(ctx);
    if (!in || !out || !min || !max || in == out || inc < 1) return set_error(ctx, MVSIM_EINVAL, "dev_extract_interval: bad argument");
    for (int d = 0; d < 3; ++d)
        if (min[d] < 0 || max[d] >= in->dims[d] || min[d] > max[d])
            return set_error(ctx, MVSIM_EINVAL, "dev_extract_interval: interval must satisfy 0 <= min <= max < dims");
    if (out->dims[0] != max[0] - min[0] + 1 || out->dims[1] != max[1] - min[1] + 1 || out->dims[2] != (max[2] - min[2]) / inc + 1)
        return set_error(ctx, MVSIM_EINVAL, "dev_extract_interval: out dims must be (max0-min0+1, max1-min1+1, (max2-min2)/inc+1)");
    StageTimer t(ctx, MVSIM_T_SAMPLE);
    return k_extract_interval(ctx, in->d, in->dims, min, max, inc, snr, seed, stream, out->d);
}

int mvsim_dev_simulate_view(mvsim_ctx* ctx, const mvsim_view_params* p, const mvsim_volume* gt, mvsim_volume* psf, mvsim_volume* out)
{
    MVSIM_ENTER(ctx);
    MVSIM_TRY(check_view(ctx, p));
    if (!gt || !psf || !out) return set_error(ctx, MVSIM_EINVAL, "dev_simulate_view: null volume");
    for (int d = 0; d < 3; ++d)
        if (gt->dims[d] != p->dims[d] || psf->dims[d] != p->kdims[d]) return set_error(ctx, MVSIM_EINVAL, "dev_simulate_view: params do not match the volumes");
    if (out->dims[0] != p->dims[0] || out->dims[1] != p->dims[1] || out->dims[2] != kept_planes(p->dims, p->inc))
        return set_error(ctx, MVSIM_EINVAL, "dev_simulate_view: out dims must be (X, Y, (Z-1)/inc+1)");
    return dev_simulate_view(ctx, p, gt->d, psf->d, out->d);
}

// ---- main()'s aligned outputs (:588-663) -------------------------------------------------------------------------------
static int check_view_list(mvsim_ctx* ctx, int n_all, int n, const int32_t* views, const char* what)
{
    if (n_all < 1 || n_all > MVSIM_MAX_WEIGHT_VIEWS) return set_error(ctx, MVSIM_EINVAL, "%s: n_all must be 1..%d", what, MVSIM_MAX_WEIGHT_VIEWS);
    if (n < 0 || n > n_all || (n > 0 && !views)) return set_error(ctx, MVSIM_EINVAL, "%s: 0..n_all view indices", what);
    bool seen[MVSIM_MAX_WEIGHT_VIEWS] = {};
    for (int i = 0; i < n; ++i) {
        if (views[i] < 0 || views[i] >= n_all) return set_error(ctx, MVSIM_EINVAL, "%s: view index %d out of range", what, (int)views[i]);
        if (seen[views[i]]) return set_error(ctx, MVSIM_EINVAL, "%s: view index %d repeated", what, (int)views[i]);
        seen[views[i]] = true;
    }
    return MVSIM_OK;
}

// axis-0 inverses of all views for the weight dims (n_all x 12)
static void weight_inverses(const int64_t dims[3], int n_all, const int32_t* align_degrees, double* inv)
{
    for (int k = 0; k < n_all; ++k) axis_rotation(dims, 0, align_degrees[k], nullptr, inv + 12 * k);
}

static int dev_align_view(mvsim_ctx* ctx, const float* acq, const int64_t acq_dims[3], int inc, int degrees, float* out)
{
    // the inverse affine of the isotropic dims, as rotateAroundAxis(iso, 0, degrees) computes it (:591); about x its row 0 is the
    // identity, which is what lets the gather follow rotate_axis0_kernel
    const int64_t iso[3] = { acq_dims[0], acq_dims[1], (acq_dims[2] - 1) * inc + 1 };
    double inv[12];
    axis_rotation(iso, 0, degrees, nullptr, inv);
    return k_align_view(ctx, acq, acq_dims, inc, inv, out);
}

int mvsim_dev_align_view(mvsim_ctx* ctx, const mvsim_volume* acq, int inc, int degrees, mvsim_volume* out)
{
    MVSIM_ENTER(ctx);
    if (!acq || !out || acq == out || inc < 1) return set_error(ctx, MVSIM_EINVAL, "dev_align_view: bad argument");
    const int64_t iso[3] = { acq->dims[0], acq->dims[1], (acq->dims[2] - 1) * inc + 1 };
    MVSIM_TRY(check_dims(ctx, iso, "dev_align_view"));
    if (out->dims[0] != iso[0] || out->dims[1] != iso[1] || out->dims[2] != iso[2])
        return set_error(ctx, MVSIM_EINVAL, "dev_align_view: out dims must be (X, Y, (Za-1)*inc+1)");
    return dev_align_view(ctx, acq->d, acq->dims, inc, degrees, out->d);
}

int mvsim_dev_aligned_weights(mvsim_ctx* ctx, const int64_t dims[3], int n_all, const int32_t* align_degrees, float osem,
                              int n_out, const int32_t* views, mvsim_volume* const* out, mvsim_volume* sum_weights)
{
    MVSIM_ENTER(ctx);
    MVSIM_TRY(check_dims(ctx, dims, "dev_aligned_weights"));
    MVSIM_TRY(check_view_list(ctx, n_all, n_out, views, "dev_aligned_weights"));
    if (!align_degrees || (n_out > 0 && !out)) return set_error(ctx, MVSIM_EINVAL, "dev_aligned_weights: null argument");
    float* d[MVSIM_MAX_WEIGHT_VIEWS] = {};
    for (int j = 0; j < n_out; ++j) {
        const mvsim_volume* o = out[j];
        if (!o || o->dims[0] != dims[0] || o->dims[1] != dims[1] || o->dims[2] != dims[2])
            return set_error(ctx, MVSIM_EINVAL, "dev_aligned_weights: output %d must be a volume of dims", j);
        d[j] = o->d;
    }
    if (sum_weights && (sum_weights->dims[0] != dims[0] || sum_weights->dims[1] != dims[1] || sum_weights->dims[2] != dims[2]))
        return set_error(ctx, MVSIM_EINVAL, "dev_aligned_weights: sum_weights must be a volume of dims");
    double inv[12 * MVSIM_MAX_WEIGHT_VIEWS];
    weight_inverses(dims, n_all, align_degrees, inv);
    return k_aligned_weights(ctx, dims, n_all, inv, osem, n_out, views, d, sum_weights ? sum_weights->d : nullptr);
}

// main()'s view loop with its post-acquisition chain (:567-663).  Per view: the whole-view acquisition (dev_simulate_view), then the
// aligned view, the view's own normalised weights and the rotated-back PSF, into one of TWO device output sets; the downloads of
// view i run on the copy stream under the kernels of view i + 1, and view i + 2 waits for them before it reuses the set.
static int simulate_dataset_impl(mvsim_ctx* ctx, int n_all, const mvsim_view_params* params, const int32_t* align_degrees, float osem,
                                 int n_views, const int32_t* views, const float* gt, const mvsim_volume* vol, float* const* psfs,
                                 const mvsim_dataset_outputs* outs, float* sum_weights)
{
    MVSIM_TRY(check_view_list(ctx, n_all, n_views, views, "simulate_dataset"));
    if (!params || !align_degrees) return set_error(ctx, MVSIM_EINVAL, "simulate_dataset: null params or angles");
    MVSIM_TRY(check_views(ctx, n_all, params, vol, "simulate_dataset"));
    for (int k = 0; k < n_all; ++k)
        if (params[k].axis != 0) return set_error(ctx, MVSIM_EINVAL, "simulate_dataset: main() rotates about x only (axis 0)");
    if (n_views > 0 && (!psfs || !outs || (!gt && !vol))) return set_error(ctx, MVSIM_EINVAL, "simulate_dataset: null argument");
    for (int i = 0; i < n_views; ++i)
        if (!psfs[i]) return set_error(ctx, MVSIM_EINVAL, "simulate_dataset: null PSF for view %d", (int)views[i]);
    if (n_views == 0 && !sum_weights) return MVSIM_OK;
    const int64_t* dims = params[0].dims;
    const size_t n = elems(dims);
    double inv_w[12 * MVSIM_MAX_WEIGHT_VIEWS];
    weight_inverses(dims, n_all, align_degrees, inv_w);
    auto iso_elems = [&](const mvsim_view_params* p) { return (size_t)(p->dims[0] * p->dims[1] * ((kept_planes(p->dims, p->inc) - 1) * p->inc + 1)); };
    // sizes of a device output set: the largest of its views
    size_t acq_max = 0, iso_max = 0, k_max = 0;
    bool any_iso = false, any_kpsf = false, any_w = false;
    for (int i = 0; i < n_views; ++i) {
        const mvsim_view_params* p = &params[views[i]];
        acq_max = std::max(acq_max, kept_elems(p->dims, p->inc));
        iso_max = std::max(iso_max, iso_elems(p));
        k_max = std::max(k_max, elems(p->kdims));
        any_iso |= outs[i].aligned != nullptr;
        any_kpsf |= outs[i].aligned_psf != nullptr;
        any_w |= outs[i].weights != nullptr;
    }
    BatchCall bc(ctx, "simulate_dataset");
    const cudaEvent_t done[2] = { bc.event(), bc.event() }, freed[2] = { bc.event(), bc.event() };
    const float* gt_dev = n_views > 0 ? bc.ground_truth(gt, vol, n) : nullptr;
    std::vector<float*> kpsf((size_t)n_views, nullptr);
    for (int i = 0; i < n_views; ++i) kpsf[(size_t)i] = bc.alloc<float>(elems(params[views[i]].kdims));
    struct OutSet { float *acq, *iso, *kpsf, *w; } set[2] = {};
    for (int s = 0; s < 2 && s < n_views; ++s) {
        set[s].acq = bc.alloc<float>(acq_max);
        if (any_iso) set[s].iso = bc.alloc<float>(iso_max);
        if (any_kpsf) set[s].kpsf = bc.alloc<float>(k_max);
        if (any_w) set[s].w = bc.alloc<float>(n);
    }
    float* dsum = sum_weights ? bc.alloc<float>(n) : nullptr;
    // downloads of view i (psfs are normalised in place, :255)
    auto download = [&](int i) -> int {
        const int s = i % 2;
        const mvsim_view_params* p = &params[views[i]];
        const mvsim_dataset_outputs& o = outs[i];
        cudaError_t e = cudaStreamWaitEvent(ctx->copy_stream, done[s], 0);
        if (e == cudaSuccess) e = cudaMemcpyAsync(psfs[i], kpsf[(size_t)i], elems(p->kdims) * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_stream);
        if (e == cudaSuccess && o.acq) e = cudaMemcpyAsync(o.acq, set[s].acq, kept_elems(p->dims, p->inc) * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_stream);
        if (e == cudaSuccess && o.aligned) e = cudaMemcpyAsync(o.aligned, set[s].iso, iso_elems(p) * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_stream);
        if (e == cudaSuccess && o.aligned_psf) e = cudaMemcpyAsync(o.aligned_psf, set[s].kpsf, elems(p->kdims) * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_stream);
        if (e == cudaSuccess && o.weights) e = cudaMemcpyAsync(o.weights, set[s].w, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_stream);
        if (e == cudaSuccess) e = cudaEventRecord(freed[s], ctx->copy_stream);
        return e == cudaSuccess ? MVSIM_OK : cuda_fail(ctx, e, "simulate_dataset: download");
    };
    if (n_views > 0)
        bc.upload([&]() -> int {
            int st = MVSIM_OK;
            for (int i = 0; i < n_views && st == MVSIM_OK; ++i) st = h2d(ctx, kpsf[(size_t)i], psfs[i], elems(params[views[i]].kdims) * sizeof(float));
            return st;
        });
    bc.compute([&](cudaEvent_t* last) -> int {
        int st = MVSIM_OK;
        // the sum image depends on the dims and the angles alone (:648-663)
        if (dsum) st = k_aligned_weights(ctx, dims, n_all, inv_w, osem, 0, nullptr, nullptr, dsum);
        for (int i = 0; i < n_views && st == MVSIM_OK; ++i) {
            const int s = i % 2, v = views[i];
            const mvsim_view_params* p = &params[v];
            const mvsim_dataset_outputs& o = outs[i];
            if (i >= 2 && cudaStreamWaitEvent(ctx->stream, freed[s], 0) != cudaSuccess) { st = set_error(ctx, MVSIM_ECUDA, "simulate_dataset: wait"); break; }
            if ((st = dev_simulate_view(ctx, p, gt_dev, kpsf[(size_t)i], set[s].acq)) != MVSIM_OK) break;                 // :570-585
            const int64_t acq_dims[3] = { p->dims[0], p->dims[1], kept_planes(p->dims, p->inc) };
            if (o.aligned && (st = dev_align_view(ctx, set[s].acq, acq_dims, p->inc, align_degrees[v], set[s].iso)) != MVSIM_OK) break;   // :588, :591
            if (o.weights && (st = k_aligned_weights(ctx, dims, n_all, inv_w, osem, 1, &v, &set[s].w, nullptr)) != MVSIM_OK) break;      // :576, :592, :615-646
            if (o.aligned_psf && (st = dev_rotate(ctx, kpsf[(size_t)i], set[s].kpsf, p->kdims, 0, align_degrees[v])) != MVSIM_OK) break; // :593
            if (cudaEventRecord(done[s], ctx->stream) != cudaSuccess) { st = set_error(ctx, MVSIM_ECUDA, "simulate_dataset: event"); break; }
            if (i >= 1) st = download(i - 1);
        }
        if (st == MVSIM_OK && n_views > 0) st = download(n_views - 1);
        if (st == MVSIM_OK && dsum) st = d2h(ctx, sum_weights, dsum, n * sizeof(float));
        *last = n_views > 0 ? done[(n_views - 1) % 2] : nullptr;
        return st;
    });
    return bc.finish();
}

int mvsim_simulate_dataset(mvsim_ctx* ctx, int n_all, const mvsim_view_params* params, const int32_t* align_degrees, float osem,
                           int n_views, const int32_t* views, const float* gt, float* const* psfs, const mvsim_dataset_outputs* outs,
                           float* sum_weights)
{
    MVSIM_ENTER(ctx);
    return simulate_dataset_impl(ctx, n_all, params, align_degrees, osem, n_views, views, gt, nullptr, psfs, outs, sum_weights);
}

int mvsim_dev_simulate_dataset(mvsim_ctx* ctx, int n_all, const mvsim_view_params* params, const int32_t* align_degrees, float osem,
                               int n_views, const int32_t* views, const mvsim_volume* gt, float* const* psfs,
                               const mvsim_dataset_outputs* outs, float* sum_weights)
{
    MVSIM_ENTER(ctx);
    return simulate_dataset_impl(ctx, n_all, params, align_degrees, osem, n_views, views, nullptr, gt, psfs, outs, sum_weights);
}


// ---- the rest of the loop body (:570-585) for ONE view whose volume is decomposed by z slabs over ranks (BASELINE config 5) ------
// convolve is mvsim_slabconv_*; these are the stages around it.  All pointers are DEVICE pointers.
int mvsim_slab_rotate_attenuate(mvsim_ctx* ctx, const float* d_gt, const int64_t dims[3], int axis, int degrees, double delta, int strict_reference,
                                int64_t z0, int64_t z_local, float* d_out_slab)
{
    MVSIM_ENTER(ctx);
    if (!d_gt || !d_out_slab) return set_error(ctx, MVSIM_EINVAL, "slab_rotate_attenuate: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "slab_rotate_attenuate"));
    if (z0 < 0 || z_local < 1 || z0 + z_local > dims[2]) return set_error(ctx, MVSIM_EINVAL, "slab_rotate_attenuate: slab outside the volume");
    if (axis < 0 || axis > 2) return set_error(ctx, MVSIM_EINVAL, "slab_rotate_attenuate: axis must be 0, 1 or 2");
    const int st = dev_rotate_attenuate(ctx, d_gt, d_out_slab, dims, axis, degrees, delta, strict_reference, z0, z_local);
    if (st == MVSIM_EUNSUPPORTED) return set_error(ctx, MVSIM_EUNSUPPORTED, "slab_rotate_attenuate: only rotations about axis 0 (the reference's) are decomposed");
    return st;
}

int mvsim_slab_sum(mvsim_ctx* ctx, const float* d_slab, size_t n_local, double* d_sum)
{
    MVSIM_ENTER(ctx);
    if (!d_slab || !d_sum) return set_error(ctx, MVSIM_EINVAL, "slab_sum: null buffer");
    StageTimer t(ctx, MVSIM_T_ADJUST);
    return k_sum(ctx, d_slab, n_local, d_sum);
}

int mvsim_slab_adjust(mvsim_ctx* ctx, float* d_slab, size_t n_local, const double* d_sums, int world, double n_global, float min_value, float target_avg)
{
    MVSIM_ENTER(ctx);
    if (!d_slab || !d_sums || world < 1 || !(n_global >= 1)) return set_error(ctx, MVSIM_EINVAL, "slab_adjust: bad argument");
    StageTimer t(ctx, MVSIM_T_ADJUST);
    MVSIM_TRY(k_adjust_corr_ranks(ctx, d_sums, world, n_global, min_value, target_avg, ctx->d_scalars + 2));
    return k_adjust_apply(ctx, d_slab, n_local, ctx->d_scalars + 2, min_value);
}

int mvsim_slab_extract(mvsim_ctx* ctx, const float* d_slab, const int64_t dims[3], int64_t z0, int64_t z_local, int inc, float snr, uint64_t seed,
                       uint64_t stream, float* d_out, int64_t* planes_out)
{
    MVSIM_ENTER(ctx);
    if (!d_slab || !d_out) return set_error(ctx, MVSIM_EINVAL, "slab_extract: null buffer");
    MVSIM_TRY(check_dims(ctx, dims, "slab_extract"));
    if (inc < 1 || z0 < 0 || z_local < 1 || z0 + z_local > dims[2]) return set_error(ctx, MVSIM_EINVAL, "slab_extract: bad slab or inc");
    StageTimer t(ctx, MVSIM_T_SAMPLE);
    return k_extract_slab(ctx, d_slab, dims, z0, z_local, inc, nullptr, 0.f, snr, seed, stream, d_out, planes_out);
}

}  // extern "C"
