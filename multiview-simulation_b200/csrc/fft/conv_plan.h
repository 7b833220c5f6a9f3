// Host-side planning of the FFT convolution: padded sizes, the (A, B) split of every line length,
// margins and crop offsets.  Pure C++ (shared by the CUDA driver and the CPU emulation tests).
//
// Replaces the size/padding logic of imglib2-algorithm FFTConvolution.convolve()
// (FFTMethods.dimensionsRealToComplexFast + paddingIntervalCentered; reference call site
// S/SimulateMultiViewDataset.java:257-261).  The result inside the original interval does not
// depend on the padded size as long as it is >= dim + kdim - 1 (SURVEY.md appendix A.6), so the
// sizes here are chosen for the GPU: products A*B with A, B <= 40 held in registers.
#pragma once
#include <stdint.h>

namespace mvsim {

struct FftSize { int n, a, b; };

// x passes: rows per CTA = thread target / threads per line.  Measured on B200 at config 3 (576-point rows, 24 threads per line,
// profiles/r02_notes.md): the forward pass wants ~120 registers and spills under the 80-register cap of 3 CTAs x 10 rows; 6 rows x
// 4 CTAs per SM (96 registers) 0.962 -> 0.920 ms.  The inverse pass: 10 rows x 3 CTAs 0.252 ms, 6 x 4 0.277; after its stores moved to
// immediate offsets (80 registers without the address arithmetic) 10 x 3 0.238, 8 rows x 4 CTAs 0.229 ms (fft_group.cu: min_blocks).
// (forward geometry measured again after the address-arithmetic change: 5 rows 0.844, 6 rows 0.837, 8 rows x 4 CTAs 0.865 ms)
constexpr int kXThreadsFwd = 144, kXThreadsInv = 192;
constexpr int x_rows_for(int target, int a, int b) { return (target / (a > b ? a : b)) > 0 ? target / (a > b ? a : b) : 1; }
constexpr int x_rows_per_block(int a, int b, bool inverse) { return x_rows_for(inverse ? kXThreadsInv : kXThreadsFwd, a, b); }


// X(n, a, b): supported complex line lengths n = a*b, ascending; a, b are in-register sub-transform sizes
// (tools/gen_regfft.py).  Balanced splits (a ~ b) keep all threads of a line busy in both halves of the
// two-level transform, so the planner prefers e.g. 648 = 24*27 over 640 = 20*32 for a 639-point minimum.
#define MVSIM_FFT_SIZES_SMALL(X) \
    X(16, 4, 4) X(20, 4, 5) X(24, 4, 6) X(30, 5, 6) X(32, 4, 8) X(36, 6, 6) X(40, 5, 8) X(48, 6, 8) X(54, 6, 9) X(64, 8, 8) \
    X(72, 8, 9) X(80, 8, 10) X(90, 9, 10) X(100, 10, 10) X(108, 9, 12) X(120, 10, 12)
#define MVSIM_FFT_SIZES_G1(X) \
    X(128, 8, 16) X(135, 9, 15) X(144, 12, 12) X(160, 10, 16) X(180, 12, 15) X(192, 12, 16) X(216, 12, 18) X(225, 15, 15) \
    X(240, 15, 16) X(256, 16, 16) X(288, 16, 18) X(320, 16, 20) X(324, 18, 18) X(360, 18, 20)
#define MVSIM_FFT_SIZES_G2(X) \
    X(384, 16, 24) X(400, 20, 20) X(432, 18, 24) X(480, 20, 24) X(512, 16, 32) X(540, 20, 27) X(576, 24, 24) X(600, 24, 25) \
    X(625, 25, 25) X(640, 20, 32) X(648, 24, 27)
#define MVSIM_FFT_SIZES_G3(X) \
    X(675, 25, 27) X(720, 24, 30) X(729, 27, 27) X(768, 24, 32) X(810, 27, 30) X(864, 27, 32) X(900, 30, 30) \
    X(960, 30, 32)
#define MVSIM_FFT_SIZES_G4(X) \
    X(1024, 32, 32) X(1080, 30, 36) X(1152, 32, 36) X(1200, 30, 40) X(1280, 32, 40) X(1296, 36, 36) X(1440, 36, 40) \
    X(1600, 40, 40)

#ifdef MVSIM_EMU_SMALL_ONLY
// CPU emulation (tests/emu): the small sizes plus the z-line lengths of the BASELINE configs (360: configs 1 / 4 at inc 3,
// 576, 640: config 3), so that the decimated fused z pass is emulated with the splits it runs with on the GPU
#define MVSIM_FFT_SIZES(X) MVSIM_FFT_SIZES_SMALL(X) X(360, 18, 20) X(576, 24, 24) X(640, 20, 32)
#else
#define MVSIM_FFT_SIZES(X) \
    MVSIM_FFT_SIZES_SMALL(X) MVSIM_FFT_SIZES_G1(X) MVSIM_FFT_SIZES_G2(X) MVSIM_FFT_SIZES_G3(X) MVSIM_FFT_SIZES_G4(X)
#endif

// the decimated and polyphase fused z kernels are built only for z lines of these lengths (build time, fft_group.cu): covers the
// BASELINE configs (339 -> 360 with inc 3, 639 -> 640 with inc 5).  Here rather than in fft_launch.h so that the CPU emulation
// (tests/emu) enumerates the same instantiations.
constexpr int kDecMinLine = 300, kDecMaxLine = 660;

// compile-time lookup in the FULL table (also under MVSIM_EMU_SMALL_ONLY): {0, 0, 0} when n is not a supported size
constexpr FftSize fft_size_lookup(int n)
{
#define MVSIM_X(n_, a_, b_) if (n == n_) return FftSize{ n_, a_, b_ };
    MVSIM_FFT_SIZES_SMALL(MVSIM_X) MVSIM_FFT_SIZES_G1(MVSIM_X) MVSIM_FFT_SIZES_G2(MVSIM_X) MVSIM_FFT_SIZES_G3(MVSIM_X) MVSIM_FFT_SIZES_G4(MVSIM_X)
#undef MVSIM_X
    return FftSize{ 0, 0, 0 };
}

inline const FftSize* fft_size_table(int* count)
{
#define MVSIM_X(n, a, b) { n, a, b },
    static const FftSize t[] = { MVSIM_FFT_SIZES(MVSIM_X) };
#undef MVSIM_X
    *count = (int)(sizeof(t) / sizeof(t[0]));
    return t;
}

// Smallest supported size >= min_n (and <= cap when cap > 0), or nullptr.  (A cost model preferring balanced
// splits, e.g. 648 = 24*27 over 640 = 20*32, was measured on B200 and lost: the radix-3 sub-transforms cost
// more than the idle threads of the unbalanced power-of-two split.)
// mult8: x rows want a multiple of 8 complex columns (64-byte aligned row pitch, whole kx tiles).
inline const FftSize* pick_fft_size(int64_t min_n, bool mult8 = false, int64_t cap = 0)
{
    int c;
    const FftSize* t = fft_size_table(&c);
    for (int i = 0; i < c; ++i) {
        if (t[i].n < min_n || (mult8 && t[i].n % 8 != 0)) continue;
        if (cap > 0 && t[i].n > cap) break;
        return &t[i];
    }
    return nullptr;
}

// How one rank of a slab-decomposed convolution sees the problem (world = 1: the whole problem).
//   z planes [z0, z0 + z_local) of the image live on this rank for the x and y passes;
//   kx tiles [tile0, tile0 + tiles_own) with ALL z planes live on it for the z pass.
struct SlabGeom {
    int rank, world;
    int z_local, z0;
    int tiles_total, tiles_own, tile0;
};

struct ConvPlan {
    int dims[3], kdims[3];  // GLOBAL volume and kernel dims
    FftSize sx, sy, sz;     // sx.n = complex length of the folded x rows (padded real length 2*sx.n); sy = one y BLOCK
    int left[3];            // padded index p holds source index p - left   (left = kdim - 1 - kdim/2)
    int crop0[3];           // output voxel o lives at padded index o + crop0 (crop0 = kdim - 1)
    int y_blocks, y_block;  // overlap-save blocks along y: block b produces output rows [b*y_block, min((b+1)*y_block, Y))
    double scale;           // 1 / (sx.n * sy.n * sz.n)

    // Workspaces.  U1/P1 are row-major in kx (written by the x pass row by row); U2/P2/H are kx-TILE-major
    // [KT][z][ky][T] (T = lanes per CTA of the strided passes): a y line tile is one contiguous chunk
    // and a z line tile strides by Ny*T elements (73 KB at config 3) instead of Ny*KXc (5.3 MB), which
    // keeps the z pass inside a few 2 MB pages and DRAM rows.
    int64_t kxc() const { return sx.n; }
    int64_t ktiles(int t) const { return (sx.n + t - 1) / t; }
    int64_t u1_elems(int z_local) const { return (int64_t)z_local * dims[1] * sx.n; }               // [Zl][Y][KXc]
    int64_t u2_elems(int t, int z_local) const { return ktiles(t) * z_local * sy.n * t; }           // [KT][Zl][Ny][T]
    int64_t h_elems(int t, int tiles_own) const { return (int64_t)tiles_own * sz.n * sy.n * t; }    // [tiles][Nz][Ny][T]
    int64_t p1_elems() const { return (int64_t)kdims[2] * kdims[1] * sx.n; }                        // [KZ][KY][KXc]
    int64_t p2_elems(int t, int tiles_own) const { return (int64_t)tiles_own * kdims[2] * sy.n * t; }   // [tiles][KZ][Ny][T]
};

inline int max_fft_line()
{
    int c;
    const FftSize* t = fft_size_table(&c);
    return t[c - 1].n;
}

// 0 ok, 1 invalid dims, 5 unsupported (too large for the size table).  max_line (tests): cap on the y line length
// that forces overlap-save blocking at small sizes; 0 = the largest table entry.
inline int make_conv_plan(const int64_t dims[3], const int64_t kdims[3], ConvPlan* p, int max_line = 0)
{
    for (int d = 0; d < 3; ++d) {
        if (dims[d] < 1 || kdims[d] < 1 || dims[d] > (1 << 30) || kdims[d] > (1 << 30)) return 1;
        p->dims[d] = (int)dims[d];
        p->kdims[d] = (int)kdims[d];
        p->left[d] = (int)(kdims[d] - 1 - kdims[d] / 2);
        p->crop0[d] = (int)(kdims[d] - 1);
    }
    const int cap = max_line > 0 ? max_line : max_fft_line();
    // y: overlap-save blocks when one padded line would exceed the table.  Every block convolves
    // y_block + KY - 1 input rows (taken from the mirror-extended volume) into y_block output rows.
    p->y_blocks = 1;
    p->y_block = (int)dims[1];
    if (dims[1] + kdims[1] - 1 > cap) {
        const int64_t room = cap - (kdims[1] - 1);
        if (room < 1) return 5;
        p->y_blocks = (int)((dims[1] + room - 1) / room);
        p->y_block = (int)((dims[1] + p->y_blocks - 1) / p->y_blocks);
    }
    const FftSize* sx = pick_fft_size((dims[0] + kdims[0] - 1 + 1) / 2, true);
    const FftSize* sy = pick_fft_size(p->y_block + kdims[1] - 1, false, cap);
    const FftSize* sz = pick_fft_size(dims[2] + kdims[2] - 1);
    if (!sx || !sy || !sz) return 5;
    p->sx = *sx; p->sy = *sy; p->sz = *sz;
    p->scale = 1.0 / ((double)sx->n * (double)sy->n * (double)sz->n);
    return 0;
}

// 0 ok, 5 when the decomposition does not divide evenly (slabs of equal size are required)
inline int make_slab_geom(const ConvPlan& pl, int lanes, int rank, int world, SlabGeom* g)
{
    const int kt = (int)pl.ktiles(lanes);
    if (world < 1 || rank < 0 || rank >= world) return 1;
    if (pl.dims[2] % world != 0 || kt % world != 0) return 5;
    g->rank = rank; g->world = world;
    g->z_local = pl.dims[2] / world; g->z0 = rank * g->z_local;
    g->tiles_total = kt; g->tiles_own = kt / world; g->tile0 = rank * g->tiles_own;
    return 0;
}

// exp(-2 pi i m / n), m < n  (double-built, float-stored) -- table for the inter-level twiddles
inline void fill_twiddles(int n, float* re_im /* 2n floats */)
{
    for (int m = 0; m < n; ++m) {
        const double a = -2.0 * 3.14159265358979323846 * (double)m / (double)n;
        re_im[2 * m] = (float)__builtin_cos(a);
        re_im[2 * m + 1] = (float)__builtin_sin(a);
    }
}
// exp(-i pi m / (2n)), m < n -- the twist of the folded real transform of padded length 2n
inline void fill_twist(int n, float* re_im)
{
    for (int m = 0; m < n; ++m) {
        const double a = -3.14159265358979323846 * (double)m / (2.0 * (double)n);
        re_im[2 * m] = (float)__builtin_cos(a);
        re_im[2 * m + 1] = (float)__builtin_sin(a);
    }
}

}  // namespace mvsim
