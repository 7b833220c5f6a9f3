// Launch interface of the line-FFT kernels.  The kernels are instantiated per supported size in
// fft_group.cu, compiled once per size group (-DMVSIM_GROUP=k) so the build parallelises.
#pragma once
#include <cuda_runtime.h>
#include "conv_plan.h"
#include "line_fft.cuh"

namespace mvsim {

enum FftKind { FFT_XFWD = 0, FFT_XINV = 1, FFT_SFWD = 2, FFT_SINV = 3, FFT_ZFUSED = 4, FFT_ZFUSED_OTF = 5,
               FFT_ZFUSED_DEC3 = 6, FFT_ZFUSED_DEC5 = 7,     // decimated inverse (ZFusedDec): the planner's (a, b) with 3 | a resp. 5 | a
               FFT_ZFUSED_POLY3 = 8, FFT_ZFUSED_POLY5 = 9 }; // polyphase form (ZFusedPoly): 3 resp. 5 phases of n / inc points

// Lanes (T) = neighbouring kx columns a CTA of the strided passes owns: 8 complex = 64-byte segments.
// (T = 4 with 4 CTAs/SM was measured on B200 and gave the same throughput; only T = 8 is built.)
int strided_lanes();

// returns cudaError_t as int, or -1 when `n` is not in this group.  One translation unit per group.
#define MVSIM_DECL(g, t) int fft_launch_g##g##_t##t(int kind, int n, const void* params, unsigned gx, unsigned gy, cudaStream_t s);
MVSIM_DECL(0, 8) MVSIM_DECL(1, 8) MVSIM_DECL(2, 8) MVSIM_DECL(3, 8) MVSIM_DECL(4, 8)
#undef MVSIM_DECL
// decimated fused z kernels (kinds FFT_ZFUSED_DEC*): line lengths kDecMinLine..kDecMaxLine live in groups 1 and 2
int fft_launch_dec_g1_t8(int kind, int n, const void* params, unsigned gx, unsigned gy, cudaStream_t s);
int fft_launch_dec_g2_t8(int kind, int n, const void* params, unsigned gx, unsigned gy, cudaStream_t s);
// polyphase fused z kernels (kinds FFT_ZFUSED_POLY*), same line lengths, their own translation units
int fft_launch_poly_g1_t8(int kind, int n, const void* params, unsigned gx, unsigned gy, cudaStream_t s);
int fft_launch_poly_g2_t8(int kind, int n, const void* params, unsigned gx, unsigned gy, cudaStream_t s);

inline int fft_launch(int kind, int lanes, int n, const void* params, unsigned gx, unsigned gy, cudaStream_t s)
{
    (void)lanes;
    if (kind >= FFT_ZFUSED_POLY3) {
        int d = fft_launch_poly_g1_t8(kind, n, params, gx, gy, s);
        if (d == -1) d = fft_launch_poly_g2_t8(kind, n, params, gx, gy, s);
        return d;
    }
    if (kind >= FFT_ZFUSED_DEC3) {
        int d = fft_launch_dec_g1_t8(kind, n, params, gx, gy, s);
        if (d == -1) d = fft_launch_dec_g2_t8(kind, n, params, gx, gy, s);
        return d;
    }
    int r = fft_launch_g0_t8(kind, n, params, gx, gy, s);
    if (r == -1) r = fft_launch_g1_t8(kind, n, params, gx, gy, s);
    if (r == -1) r = fft_launch_g2_t8(kind, n, params, gx, gy, s);
    if (r == -1) r = fft_launch_g3_t8(kind, n, params, gx, gy, s);
    if (r == -1) r = fft_launch_g4_t8(kind, n, params, gx, gy, s);
    return r;
}

}  // namespace mvsim
