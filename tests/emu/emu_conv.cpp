// CPU emulation of the CUDA line-FFT kernels: runs the very same __host__ __device__ phase
// functions (multiview-simulation_b200/csrc/fft/line_fft.cuh) thread by thread, block by block,
// with a barrier between phases, driven by the same host logic (conv_driver.h).  Built with g++
// by tests/test_emu_conv.py (the small size table) and tests/test_emu_fft_sizes.py (-DMVSIM_EMU_FULL_TABLE: every
// line length the library ships); this is a test of the index arithmetic, not a product path.
#ifndef MVSIM_EMU_FULL_TABLE
#define MVSIM_EMU_SMALL_ONLY 1
#endif
#define MVSIM_PACKED_FFT 1
#include "fft/conv_driver.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <vector>

using namespace mvsim;

// dynamic shared memory of a launch: K::SMEM_BYTES, or K::smem_bytes(params) where the kernel sizes an area at run time
template <class K, class = void> struct EmuSmem { static size_t bytes(const typename K::Params&) { return (size_t)K::SMEM_BYTES; } };
template <class K> struct EmuSmem<K, std::void_t<decltype(&K::smem_bytes)>> {
    static size_t bytes(const typename K::Params& q) { return (size_t)K::smem_bytes(q); }
};

template <class K> static void emulate(const typename K::Params& q, int gx, int gy)
{
    std::vector<float2> sm(EmuSmem<K>::bytes(q) / sizeof(float2) + 8);
    std::vector<typename K::State> st(K::THREADS);
    for (int by = 0; by < gy; ++by)
        for (int bx = 0; bx < gx; ++bx) {
            // poison shared memory so stale reads show up
            for (auto& v : sm) { v.x = 1e30f; v.y = -1e30f; }
            for (int t = 0; t < K::THREADS; ++t) K::template phase<0>(q, bx, by, t, sm.data(), st[t]);
            if (K::NPH > 1) for (int t = 0; t < K::THREADS; ++t) K::template phase<1>(q, bx, by, t, sm.data(), st[t]);
            if (K::NPH > 2) for (int t = 0; t < K::THREADS; ++t) K::template phase<2>(q, bx, by, t, sm.data(), st[t]);
            if (K::NPH > 3) for (int t = 0; t < K::THREADS; ++t) K::template phase<3>(q, bx, by, t, sm.data(), st[t]);
            if (K::NPH > 4) for (int t = 0; t < K::THREADS; ++t) K::template phase<4>(q, bx, by, t, sm.data(), st[t]);
            if (K::NPH > 5) for (int t = 0; t < K::THREADS; ++t) K::template phase<5>(q, bx, by, t, sm.data(), st[t]);
            if (K::NPH > 6) for (int t = 0; t < K::THREADS; ++t) K::template phase<6>(q, bx, by, t, sm.data(), st[t]);
            if (K::NPH > 7) for (int t = 0; t < K::THREADS; ++t) K::template phase<7>(q, bx, by, t, sm.data(), st[t]);
        }
}

static constexpr int T = 8;
// x_rows_per_block (fft/conv_plan.h): the emulation uses the CUDA launcher's rows per CTA
template <int A, int B> struct Rows { static constexpr int RF = x_rows_per_block(A, B, false), RI = x_rows_per_block(A, B, true); };

struct EmuLauncher {
    int lanes = T;
    bool h_on_the_fly = false;
    int x_blocks(const FftSize& s, int n_rows, bool inverse) const
    {
        const int r = x_rows_per_block(s.a, s.b, inverse);
        return (n_rows + r - 1) / r;
    }
    int launch_x(bool inverse, const FftSize& s, const XParams& q)
    {
        const int gx = x_blocks(s, q.n_rows, inverse);
        switch (s.n) {
#define MVSIM_X(n_, a_, b_) case n_: if (inverse) emulate<XInv<a_, b_, Rows<a_, b_>::RI>>(q, gx, 1); else emulate<XFwd<a_, b_, Rows<a_, b_>::RF>>(q, gx, 1); return 0;
            MVSIM_FFT_SIZES(MVSIM_X)
#undef MVSIM_X
        }
        return 5;
    }
    int launch_strided(bool inverse, const FftSize& s, const StridedParams& q0, int tiles, int n_outer)
    {
        StridedParams q = q0;
        strided_fill_e32(q, s.n);
        const int gx = q.swap_grid ? n_outer : tiles, gy = q.swap_grid ? tiles : n_outer;
        switch (s.n) {
#define MVSIM_X(n_, a_, b_) case n_: if (inverse) emulate<StridedInv<a_, b_, T>>(q, gx, gy); else emulate<StridedFwd<a_, b_, T>>(q, gx, gy); return 0;
            MVSIM_FFT_SIZES(MVSIM_X)
#undef MVSIM_X
        }
        return 5;
    }
    bool z_decimate(const FftSize&) const { return getenv("MVSIM_EMU_DECIMATE") != nullptr; }
    int launch_zfused_dec(const FftSize& s, const ZFusedParams& q0, int tiles, int n_outer, int inc)
    {
        ZFusedParams q = q0;
        std::vector<float2> d((size_t)s.n);
        zfused_dec_table(s.n, q.crop0, q.n_src, inc, d.data());
        q.dtab = d.data();
        ++decimated_launches;
        switch (s.n) {
#define MVSIM_X(n_, a_, b_) case n_: return inc == 3 ? dec<a_, b_, 3>(q, n_outer, tiles) : dec<a_, b_, 5>(q, n_outer, tiles);

            MVSIM_FFT_SIZES(MVSIM_X)
#undef MVSIM_X
        }
        return 5;
    }
    template <int A, int B, int INC> static int dec(const ZFusedParams& q, int n_outer, int tiles)
    {
        if constexpr (zfused_dec_ok(A, B, INC)) {
            emulate<ZFusedDec<B, A, T, INC>>(q, n_outer, tiles);
            return 0;
        } else {
            return 5;
        }
    }
    static int decimated_launches;
    // polyphase form of the whole-view fused z pass (ZFusedPoly)
    bool z_polyphase(const FftSize& s, int inc, int k_src) const { return getenv("MVSIM_EMU_POLY") != nullptr && k_src <= zfused_poly_max_taps(s.n, inc); }
    int launch_zfused_poly(const FftSize& s, const ZFusedParams& q, int tiles, int n_outer, int inc)
    {
        ++polyphase_launches;
        switch (s.n) {
#define MVSIM_X(n_, a_, b_) case n_: return inc == 3 ? poly<n_, 3>(q, n_outer, tiles) : poly<n_, 5>(q, n_outer, tiles);
            MVSIM_FFT_SIZES(MVSIM_X)
#undef MVSIM_X
        }
        return 5;
    }
    template <int N, int INC> static int poly(const ZFusedParams& q, int n_outer, int tiles)
    {
        if constexpr (zfused_poly_ok(N, INC)) {
            emulate<ZFusedPoly<N, INC, T>>(q, n_outer, tiles);
            return 0;
        } else {
            return 5;
        }
    }
    static int polyphase_launches;
    int launch_zfused(const FftSize& s, const ZFusedParams& q, int tiles, int n_outer)
    {
        if (q.h_mode)
            switch (s.n) {
#define MVSIM_X(n_, a_, b_) case n_: emulate<ZFusedOTF<a_, b_, T>>(q, n_outer, tiles); return 0;
                MVSIM_FFT_SIZES(MVSIM_X)
#undef MVSIM_X
            }
        switch (s.n) {
#define MVSIM_X(n_, a_, b_) case n_: emulate<ZFused<a_, b_, T>>(q, n_outer, tiles); return 0;
            MVSIM_FFT_SIZES(MVSIM_X)
#undef MVSIM_X
        }
        return 5;
    }
};

int EmuLauncher::decimated_launches = 0;
extern "C" int emu_decimated_launches() { return EmuLauncher::decimated_launches; }
// which (line length, inc) pairs the polyphase fused z kernel is built for (fft_group.cu), and how many PSF taps its border groups take
extern "C" int emu_poly_ok(int n, int inc)
{
    const bool built = n >= kDecMinLine && n <= kDecMaxLine && fft_size_lookup(n).n == n;
    return (built && n % inc == 0 && zfused_poly_ok(n, inc)) ? zfused_poly_max_taps(n, inc) : 0;
}
// which (line length, inc) pairs the decimated fused z kernel is built for (fft_group.cu: ZFusedDec<b, a, T, inc> of the split n = a * b)
extern "C" int emu_dec_ok(int n, int inc)
{
    const FftSize s = fft_size_lookup(n);
    return (n >= kDecMinLine && n <= kDecMaxLine && s.n == n && zfused_dec_ok(s.a, s.b, inc)) ? 1 : 0;
}
int EmuLauncher::polyphase_launches = 0;
extern "C" int emu_polyphase_launches() { return EmuLauncher::polyphase_launches; }

extern "C" int emu_plan(const int64_t dims[3], const int64_t kdims[3], int out[11], int max_line)
{
    ConvPlan pl;
    const int err = make_conv_plan(dims, kdims, &pl, max_line);
    if (err) return err;
    out[0] = pl.sx.n; out[1] = pl.sy.n; out[2] = pl.sz.n;
    out[3] = pl.sx.a; out[4] = pl.sx.b; out[5] = pl.sy.a; out[6] = pl.sy.b; out[7] = pl.sz.a; out[8] = pl.sz.b;
    out[9] = pl.y_blocks; out[10] = pl.y_block;
    return 0;
}

static int last_sum_plane_is_total = 0;
// 1: the extra plane of the last emu_convolve(keep_inc > 1) carries the sum of ALL cropped planes (polyphase kernel), 0: of the dropped ones
extern "C" int emu_last_sum_plane_is_total() { return last_sum_plane_is_total; }

namespace {

struct RankState {
    SlabGeom g;
    std::vector<float2> u1, u1o, u2, ex, h, p1, p2;
    ConvWorkspace ws;
};

void poison(std::vector<float2>& v) { for (auto& e : v) { e.x = 3e30f; e.y = -3e30f; } }

}  // namespace

// Emulates `world` ranks of the slab-decomposed convolution in one process (world = 1: the single-GPU path).
// The all-to-all exchanges are done here on the host with the semantics of all_to_all_single (equal chunks).
// psf must already be normalised.  keep_inc > 1 (world 1 only): out receives the kept slices then the sum plane.
// p2p != 0 (world > 1): no exchange pass at all -- the y forward pass and the fused z pass store straight into the
// owners' buffers through pointer tables (on the GPU: peer memory over NVLink)
extern "C" int emu_convolve(const float* img, const int64_t dims[3], const float* psf, const int64_t kdims[3],
                            float* out, double* sum_out, int keep_inc, int world, int max_line, int p2p)
{
    ConvPlan pl;
    int err = make_conv_plan(dims, kdims, &pl, max_line);
    if (err) return err;
    std::vector<float2> twx(pl.sx.n), twy(pl.sy.n), twz(pl.sz.n), twist(pl.sx.n);
    fill_twiddles(pl.sx.n, &twx[0].x);
    fill_twiddles(pl.sy.n, &twy[0].x);
    fill_twiddles(pl.sz.n, &twz[0].x);
    fill_twist(pl.sx.n, &twist[0].x);
    EmuLauncher l;
    l.h_on_the_fly = getenv("MVSIM_EMU_OTF") != nullptr;
    std::vector<RankState> rk(world);
    for (int r = 0; r < world; ++r) {
        RankState& s = rk[r];
        err = make_slab_geom(pl, T, r, world, &s.g);
        if (err) return err;
        s.u1.resize(pl.u1_elems(s.g.z_local)); s.u1o.resize(pl.y_blocks > 1 ? pl.u1_elems(s.g.z_local) : 0);
        s.u2.resize(pl.u2_elems(T, s.g.z_local)); s.ex.resize(world > 1 ? s.u2.size() : 0);
        s.h.resize(pl.h_elems(T, s.g.tiles_own)); s.p1.resize(pl.p1_elems()); s.p2.resize(pl.p2_elems(T, s.g.tiles_own));
        // poison the workspaces: every element that is read must have been written by a pass
        for (auto* v : { &s.u1, &s.u1o, &s.u2, &s.ex, &s.h, &s.p1, &s.p2 }) poison(*v);
        s.ws = ConvWorkspace{};
        s.ws.u1 = s.u1.data(); s.ws.u1o = pl.y_blocks > 1 ? s.u1o.data() : s.u1.data(); s.ws.u2 = s.u2.data();
        s.ws.ex = world > 1 ? s.ex.data() : s.u2.data(); s.ws.h = s.h.data(); s.ws.p1 = s.p1.data(); s.ws.p2 = s.p2.data();
        s.ws.tw_x = twx.data(); s.ws.tw_y = twy.data(); s.ws.tw_z = twz.data(); s.ws.twist_x = twist.data();
        err = conv_psf_spectrum(l, pl, s.g, s.ws, psf);
        if (err) return err;
        err = conv_forward_x(l, pl, s.g, s.ws, img + (size_t)s.g.z0 * pl.dims[1] * pl.dims[0]);
        if (err) return err;
    }
    if (p2p && world > 1)
        for (int r = 0; r < world; ++r) {
            rk[r].ws.n_peers = world;
            for (int q = 0; q < world; ++q) { rk[r].ws.peers_x[q] = rk[q].ex.data(); rk[r].ws.peers_y[q] = rk[q].u2.data(); }
        }
    const int planes = conv_out_planes(pl, rk[0].g, keep_inc);
    const size_t chunk = rk[0].u2.size() / world;
    bool sum_total = false;
    for (int b = 0; b < pl.y_blocks; ++b) {
        if (world > 1 && p2p)
            for (int r = 0; r < world; ++r) poison(rk[r].ex);     // the y passes of ALL ranks must fill every z-pass buffer
        for (int r = 0; r < world; ++r)
            if ((err = conv_forward_y(l, pl, rk[r].g, rk[r].ws, b))) return err;
        if (world > 1 && !p2p)      // all-to-all: chunk d of rank s's send buffer lands in chunk s of rank d's receive buffer
            for (int s = 0; s < world; ++s)
                for (int d = 0; d < world; ++d)
                    std::memcpy(rk[d].ex.data() + s * chunk, rk[s].u2.data() + d * chunk, chunk * sizeof(float2));
        if (world > 1)
            for (int r = 0; r < world; ++r) poison(rk[r].u2);     // everything the inverse reads must arrive again
        for (int r = 0; r < world; ++r)
            if ((err = conv_middle_z(l, pl, rk[r].g, rk[r].ws, rk[r].ws.ex, keep_inc, &sum_total))) return err;
        if (world > 1 && !p2p)
            for (int s = 0; s < world; ++s)
                for (int d = 0; d < world; ++d)
                    std::memcpy(rk[d].u2.data() + s * chunk, rk[s].ex.data() + d * chunk, chunk * sizeof(float2));
        for (int r = 0; r < world; ++r)
            if ((err = conv_inverse_y(l, pl, rk[r].g, rk[r].ws, b, planes))) return err;
    }
    double total = 0;
    for (int r = 0; r < world; ++r) {
        std::vector<double> partials(l.x_blocks(pl.sx, pl.dims[1] * planes, true), 0.0);
        float* o = out + (size_t)(world > 1 ? rk[r].g.z0 : 0) * pl.dims[1] * pl.dims[0];
        if ((err = conv_inverse_x(l, pl, rk[r].ws, o, partials.data(), planes, sum_total))) return err;
        for (double v : partials) total += v;
    }
    if (sum_out) *sum_out = total;
    last_sum_plane_is_total = sum_total ? 1 : 0;
    return 0;
}

// Pruned forward sub-transforms (RegFFTPZ: inputs x[K..N) known to be zero) against the full ones, every generated size.
// Returns the largest |difference| relative to the largest output magnitude.
template <int N> static double check_pruned_one()
{
    float2 a[N], b[N];
    unsigned s = 12345u + N;
    for (int i = 0; i < N; ++i) {
        s = s * 1664525u + 1013904223u; const float re = (float)(s >> 8) / 16777216.f - 0.5f;
        s = s * 1664525u + 1013904223u; const float im = (float)(s >> 8) / 16777216.f - 0.5f;
        const bool live = i < RegFFTPZ<N>::K;
        a[i] = make_float2(live ? re : 0.f, live ? im : 0.f);
        b[i] = live ? a[i] : make_float2(777.f, -777.f);        // must not be read
    }
    RegFFTP<N, -1>::run(a);
    RegFFTPZ<N>::run(b);
    double err = 0, mag = 0;
    for (int i = 0; i < N; ++i) {
        err = std::max(err, (double)std::max(std::fabs(a[i].x - b[i].x), std::fabs(a[i].y - b[i].y)));
        mag = std::max(mag, (double)std::max(std::fabs(a[i].x), std::fabs(a[i].y)));
    }
    return err / mag;
}

extern "C" double emu_check_pruned_ffts()
{
    double e = 0;
#define MVSIM_CHK(n) e = std::max(e, check_pruned_one<n>());
    MVSIM_CHK(2) MVSIM_CHK(3) MVSIM_CHK(4) MVSIM_CHK(5) MVSIM_CHK(6) MVSIM_CHK(8) MVSIM_CHK(9) MVSIM_CHK(10) MVSIM_CHK(12) MVSIM_CHK(15)
    MVSIM_CHK(16) MVSIM_CHK(18) MVSIM_CHK(20) MVSIM_CHK(24) MVSIM_CHK(25) MVSIM_CHK(27) MVSIM_CHK(30) MVSIM_CHK(32) MVSIM_CHK(36) MVSIM_CHK(40)
#undef MVSIM_CHK
    return e;
}

// One generated sub-transform on the caller's input (2n floats, interleaved re / im), for the float64 DFT comparison of
// tests/test_emu_fft_sizes.py.  family 0: RegFFT<n, dir> (scalar), 1: RegFFTP<n, dir> (packed), 2: RegFFTPZ<n> (forward transform
// of x[0..K), x[K..n) is not read; dir ignored), 3: RegFFTPD<n, dir, r> (inverse of which only o[j] = X[r + dir * j] is computed,
// into out[0..n / dir)).  Returns 0, or -1 when that variant is not generated.
template <int N, int INC, int R> static int regfft_dec(const float2 (&x)[N], float* out)
{
    if constexpr (N % INC == 0 && N / INC >= 2 && R < INC) {
        float2 o[N / INC];
        RegFFTPD<N, INC, R>::run(x, o);
        for (int j = 0; j < N / INC; ++j) { out[2 * j] = o[j].x; out[2 * j + 1] = o[j].y; }
        return 0;
    } else {
        return -1;
    }
}

template <int N> static int regfft_one(int family, int dir, int r, const float* in, float* out)
{
    float2 x[N];
    for (int i = 0; i < N; ++i) x[i] = make_float2(in[2 * i], in[2 * i + 1]);
    if (family == 3) {
        if (dir == 3) {
            switch (r) {
            case 0: return regfft_dec<N, 3, 0>(x, out);
            case 1: return regfft_dec<N, 3, 1>(x, out);
            case 2: return regfft_dec<N, 3, 2>(x, out);
            }
        } else if (dir == 5) {
            switch (r) {
            case 0: return regfft_dec<N, 5, 0>(x, out);
            case 1: return regfft_dec<N, 5, 1>(x, out);
            case 2: return regfft_dec<N, 5, 2>(x, out);
            case 3: return regfft_dec<N, 5, 3>(x, out);
            case 4: return regfft_dec<N, 5, 4>(x, out);
            }
        }
        return -1;
    }
    if (family == 2) RegFFTPZ<N>::run(x);
    else if (family == 0 && dir == -1) RegFFT<N, -1>::run(x);
    else if (family == 0 && dir == 1) RegFFT<N, 1>::run(x);
    else if (family == 1 && dir == -1) RegFFTP<N, -1>::run(x);
    else if (family == 1 && dir == 1) RegFFTP<N, 1>::run(x);
    else return -1;
    for (int i = 0; i < N; ++i) { out[2 * i] = x[i].x; out[2 * i + 1] = x[i].y; }
    return 0;
}

// the generated sub-transform sizes: SIZES of tools/gen_regfft.py (a size added there fails the DFT test until it is listed here)
#define MVSIM_REGFFT_SIZES(X) X(2) X(3) X(4) X(5) X(6) X(8) X(9) X(10) X(12) X(15) X(16) X(18) X(20) X(24) X(25) X(27) X(30) X(32) X(36) X(40)

extern "C" int emu_regfft(int family, int n, int dir, int r, const float* in, float* out)
{
    switch (n) {
#define MVSIM_X(n_) case n_: return regfft_one<n_>(family, dir, r, in, out);
        MVSIM_REGFFT_SIZES(MVSIM_X)
#undef MVSIM_X
    }
    return -1;
}

// K of RegFFTPZ<n>: the leading inputs the pruned forward transform reads (-1: no such size)
extern "C" int emu_regfft_pz_k(int n)
{
    switch (n) {
#define MVSIM_X(n_) case n_: return RegFFTPZ<n_>::K;
        MVSIM_REGFFT_SIZES(MVSIM_X)
#undef MVSIM_X
    }
    return -1;
}
