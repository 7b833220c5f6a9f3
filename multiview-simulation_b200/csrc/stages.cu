// Streaming stage kernels of the per-view pipeline (everything except the FFT passes).
// Reference bodies replaced (S = src/main/java/net/preibisch/simulation):
//   rotate     S/SimulateMultiViewDataset.java:104-135   (single-threaded cursor loop, 8 virtual gets/voxel)
//   attenuate  S/SimulateMultiViewDataset.java:318-364   (single-threaded, stride-X walk along y)
//   sums       S/Tools.java:112-132 (normImage / sumImage, mpicbg RealSum)
//   adjust     S/Tools.java:143-159
//   extract    S/SimulateMultiViewDataset.java:195-231 + Poisson S/Tools.java:73-86
// All of them are HBM-bound; threads map to x (the contiguous axis) so every warp access is a
// full 128-byte line (float4 where the row length allows).
#include <stdlib.h>

#include "ctx.h"
#include "post.cuh"
#include "sampler.cuh"

namespace mvsim {

static inline unsigned blocks_for(size_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

#define MVSIM_LAUNCH_CHECK(ctx)                                                     \
    do {                                                                            \
        (ctx)->launches++;                                                          \
        cudaError_t e__ = cudaGetLastError();                                       \
        if (e__ != cudaSuccess) return cuda_fail((ctx), e__, "kernel launch");      \
    } while (0)

// ---------------------------------------------------------------------------------------------
// rotate.  Inverse affine applied in FP64 in mpicbg's evaluation order, floor + fractional weights in
// FP64, blend in FP32 in imglib2's tap order (000,100,110,010,011,111,101,001), zero outside.
// ---------------------------------------------------------------------------------------------
template <int VEC> struct VecT;
template <> struct VecT<1> { using type = float; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

template <int VEC> __device__ __forceinline__ void vload(float (&d)[VEC], const float* p, bool ok)
{
    using V = typename VecT<VEC>::type;
    if (ok) {
        const V v = __ldg(reinterpret_cast<const V*>(p));
        const float* f = reinterpret_cast<const float*>(&v);
#pragma unroll
        for (int i = 0; i < VEC; ++i) d[i] = f[i];
    } else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) d[i] = 0.f;
    }
}

// axis 0: x_src == x (row 0 of the inverse is the identity), so the source coordinates are constant
// along a row and the gather is bilinear in (y,z): VEC contiguous voxels per thread, 4 coalesced loads.
template <int VEC> __global__ void __launch_bounds__(256) rotate_axis0_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                                            int X, int Y, int Z, Affine a)
{
    const int XV = (X + VEC - 1) / VEC;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)XV * Y * Z;
    if (idx >= total) return;
    const int xv = (int)(idx % XV);
    const long long yz = idx / XV;
    const int y = (int)(yz % Y), z = (int)(yz / Y);
    const RowTaps t = axis0_row_taps(y, z, a);
    const bool y0 = (unsigned)t.iy < (unsigned)Y, y1 = (unsigned)(t.iy + 1) < (unsigned)Y;
    const bool z0 = (unsigned)t.iz < (unsigned)Z, z1 = (unsigned)(t.iz + 1) < (unsigned)Z;
    const long long x0 = (long long)xv * VEC;
    const long long r00 = x0 + (long long)X * (t.iy + (long long)Y * t.iz);
    const long long sy = X, sz = (long long)X * Y;
    float* o = out + x0 + (long long)X * (y + (long long)Y * z);
    float t00[VEC], t10[VEC], t11[VEC], t01[VEC], r[VEC];
    vload<VEC>(t00, in + r00, y0 && z0);
    vload<VEC>(t10, in + r00 + sy, y1 && z0);
    vload<VEC>(t11, in + r00 + sy + sz, y1 && z1);
    vload<VEC>(t01, in + r00 + sz, y0 && z1);
#pragma unroll
    for (int i = 0; i < VEC; ++i) r[i] = axis0_blend(t00[i], t10[i], t11[i], t01[i], t);
    *reinterpret_cast<typename VecT<VEC>::type*>(o) = *reinterpret_cast<typename VecT<VEC>::type*>(r);
}

__global__ void __launch_bounds__(256) rotate_general_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                            int X, int Y, int Z, Affine a)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)X * Y * Z;
    if (idx >= total) return;
    const int x = (int)(idx % X);
    const long long yz = idx / X;
    const int y = (int)(yz % Y), z = (int)(yz / Y);
    const double l0 = x, l1 = y, l2 = z;
    double p[3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
        p[r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(l0, a.m[4 * r]), __dmul_rn(l1, a.m[4 * r + 1])), __dmul_rn(l2, a.m[4 * r + 2])), a.m[4 * r + 3]);
    const double f0 = floor(p[0]), f1 = floor(p[1]), f2 = floor(p[2]);
    const double w0 = p[0] - f0, w1 = p[1] - f1, w2 = p[2] - f2;
    const double w0i = 1.0 - w0, w1i = 1.0 - w1, w2i = 1.0 - w2;
    const int ix = (int)fmax(fmin(f0, 2.0e9), -2.0e9), iy = (int)fmax(fmin(f1, 2.0e9), -2.0e9), iz = (int)fmax(fmin(f2, 2.0e9), -2.0e9);
    auto tap = [&](int dx, int dy, int dz) -> float {
        const int xx = ix + dx, yy = iy + dy, zz = iz + dz;
        if ((unsigned)xx >= (unsigned)X || (unsigned)yy >= (unsigned)Y || (unsigned)zz >= (unsigned)Z) return 0.f;
        return __ldg(in + xx + (long long)X * (yy + (long long)Y * zz));
    };
    float acc = __fmul_rn(tap(0, 0, 0), (float)(w0i * w1i * w2i));
    acc = __fadd_rn(acc, __fmul_rn(tap(1, 0, 0), (float)(w0 * w1i * w2i)));
    acc = __fadd_rn(acc, __fmul_rn(tap(1, 1, 0), (float)(w0 * w1 * w2i)));
    acc = __fadd_rn(acc, __fmul_rn(tap(0, 1, 0), (float)(w0i * w1 * w2i)));
    acc = __fadd_rn(acc, __fmul_rn(tap(0, 1, 1), (float)(w0i * w1 * w2)));
    acc = __fadd_rn(acc, __fmul_rn(tap(1, 1, 1), (float)(w0 * w1 * w2)));
    acc = __fadd_rn(acc, __fmul_rn(tap(1, 0, 1), (float)(w0 * w1i * w2)));
    acc = __fadd_rn(acc, __fmul_rn(tap(0, 0, 1), (float)(w0i * w1i * w2)));
    out[idx] = acc;
}

// ---------------------------------------------------------------------------------------------
// fused rotate (axis 0) + attenuate for the whole-view entry point: the rotated volume never goes to HBM.
// A tiny pre-pass tabulates, per output row (y,z), the row taps of rotate_axis0_kernel (post.cuh); the main
// kernel marches every (x,z) column from y = Y-1 down, gathers the rotated voxel from the ground truth and
// applies the recurrence of :343-357.
// ---------------------------------------------------------------------------------------------
// rows (y, z) of the output planes [z0, z0 + Zl): entry (z - z0) * Y + y  (RowTaps, axis0_row_taps: post.cuh)
__global__ void __launch_bounds__(256) rotate_rowtable_kernel(RowTaps* __restrict__ tab, int Y, int z0, int Zl, Affine a)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)Y * Zl) return;
    tab[i] = axis0_row_taps((int)(i % Y), z0 + (int)(i / Y), a);
}

// bounds-tested march: volumes of 2^31 voxels or more, or X % 4 != 0
template <int VEC, int U> __global__ void __launch_bounds__(128) rotate_attenuate_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                                                        const RowTaps* __restrict__ tab, int X, int Y, int Z,
                                                                                        double delta, int steps, int Zl)
{
    // `in` has Z planes; `out` and `tab` cover the Zl output planes this launch owns (Zl == Z on one GPU; a z slab of the view
    // when the volume is decomposed over ranks -- the source stays whole: a rotation about x reads planes far outside the slab)
    using V = typename VecT<VEC>::type;
    const int XV = X / VEC;
    const long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= (long long)XV * Zl) return;
    const int x0 = (int)(col % XV) * VEC, z = (int)(col / XV);      // z: local plane
    const long long sy = X, sz = (long long)X * Y;
    const RowTaps* trow = tab + (long long)Y * z;
    const long long obase = x0 + sz * z;
    double n[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) n[i] = 1.0;
    int y = Y - 1, s = 0;
    // the row taps of the NEXT batch are requested while this batch's gathers are in flight: the table load sat in series with
    // the gather (ncu source view, r02a: 14 % of the stall samples on the first use of the table entry)
    RowTaps tp[U];
    if (steps >= U) {
#pragma unroll
        for (int j = 0; j < U; ++j) tp[j] = trow[y - j];
    }
    for (; s + U <= steps; s += U, y -= U) {
        float t00[U][VEC], t10[U][VEC], t11[U][VEC], t01[U][VEC];
        RowTaps tn[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int yn = y - U - j;
            tn[j] = trow[yn > 0 ? yn : 0];
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int iy = tp[j].iy, iz = tp[j].iz;
            const bool y0 = (unsigned)iy < (unsigned)Y, y1 = (unsigned)(iy + 1) < (unsigned)Y;
            const bool z0 = (unsigned)iz < (unsigned)Z, z1 = (unsigned)(iz + 1) < (unsigned)Z;
            const long long r = x0 + sy * iy + sz * iz;
            vload<VEC>(t00[j], in + r, y0 && z0);
            vload<VEC>(t10[j], in + (r + sy), y1 && z0);
            vload<VEC>(t11[j], in + (r + sy + sz), y1 && z1);
            vload<VEC>(t01[j], in + (r + sz), y0 && z1);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            float res[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) res[i] = attenuate_step(axis0_blend(t00[j][i], t10[j][i], t11[j][i], t01[j][i], tp[j]), delta, n[i]);
            *reinterpret_cast<V*>(out + (obase + sy * (y - j))) = *reinterpret_cast<V*>(res);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) tp[j] = tn[j];
    }
    for (; s < steps; ++s, --y) {
        const RowTaps t = trow[y];
        const bool y0 = (unsigned)t.iy < (unsigned)Y, y1 = (unsigned)(t.iy + 1) < (unsigned)Y;
        const bool z0 = (unsigned)t.iz < (unsigned)Z, z1 = (unsigned)(t.iz + 1) < (unsigned)Z;
        const long long r = x0 + sy * t.iy + sz * t.iz;
        float a00[VEC], a10[VEC], a11[VEC], a01[VEC], res[VEC];
        vload<VEC>(a00, in + r, y0 && z0);
        vload<VEC>(a10, in + (r + sy), y1 && z0);
        vload<VEC>(a11, in + (r + sy + sz), y1 && z1);
        vload<VEC>(a01, in + (r + sz), y0 && z1);
#pragma unroll
        for (int i = 0; i < VEC; ++i) res[i] = attenuate_step(axis0_blend(a00[i], a10[i], a11[i], a01[i], t), delta, n[i]);
        *reinterpret_cast<V*>(out + (obase + sy * y)) = *reinterpret_cast<V*>(res);
    }
    float zero[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) zero[i] = 0.f;
    for (; y >= 0; --y) *reinterpret_cast<V*>(out + (obase + sy * y)) = *reinterpret_cast<V*>(zero);
}

// The same march with the tap ADDRESSES tabulated (RowTapsOff, axis0_row_offsets: post.cuh): four unconditional float4 loads per
// row and no instruction on bounds (ncu r02c: half of the kernel's cycles issue, a quarter of its instructions were offsets, bound
// predicates and the zero fill of masked taps).  Volumes below 2^31 voxels, X % 4 == 0.
__global__ void __launch_bounds__(256) rotate_rowtable_off_kernel(RowTapsOff* __restrict__ tab, int X, int Y, int Z, int z0, int Zl, Affine a)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)Y * Zl) return;
    tab[i] = axis0_row_offsets(axis0_row_taps((int)(i % Y), z0 + (int)(i / Y), a), X, Y, Z);
}

// esz = sizeof(float) as a RUN-TIME value: tap addresses become one widening multiply-add (IMAD.WIDE.U32) each instead of the shift +
// add-with-carry pair a constant scale compiles to (the same change took the forward x pass from 0.918 to 0.836 ms)
__device__ __forceinline__ float4 tap4(const float* base, unsigned off, unsigned esz)
{
    return __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const char*>(base) + (unsigned long long)off * (unsigned long long)esz));
}

// The blend of an out-of-volume tap is f32(s * 0) with the voxel s of row (0, 0): bit-identical to rotate_attenuate_kernel for finite
// source data without negative values (RowTapsOff).  The recurrence clamps through the sign bit (clamp0): the same as fmax there.
template <int U> __global__ void __launch_bounds__(128) rotate_attenuate_off_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                                                    const RowTapsOff* __restrict__ tab, int X, int Y,
                                                                                    double delta, int steps, int Zl, unsigned esz)
{
    const int XV = X / 4;
    const long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= (long long)XV * Zl) return;
    const int x0 = (int)(col % XV) * 4, z = (int)(col / XV);      // z: local plane
    const unsigned sy = (unsigned)X;
    const RowTapsOff* trow = tab + (long long)Y * z;
    const float* src = in + x0;
    float* dst = out + (size_t)x0 + (size_t)X * Y * z;
    double n[4] = { 1.0, 1.0, 1.0, 1.0 };
    int y = Y - 1, s = 0;
    RowTapsOff tp[U];
    if (steps >= U) {
#pragma unroll
        for (int j = 0; j < U; ++j) tp[j] = trow[y - j];
    }
    for (; s + U <= steps; s += U, y -= U) {
        float4 t00[U], t10[U], t11[U], t01[U];
        RowTapsOff tn[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int yn = y - U - j;
            tn[j] = trow[yn > 0 ? yn : 0];
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            t00[j] = tap4(src, tp[j].o00, esz);
            t10[j] = tap4(src, tp[j].o10, esz);
            t11[j] = tap4(src, tp[j].o11, esz);
            t01[j] = tap4(src, tp[j].o01, esz);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const float a00[4] = { t00[j].x, t00[j].y, t00[j].z, t00[j].w }, a10[4] = { t10[j].x, t10[j].y, t10[j].z, t10[j].w };
            const float a11[4] = { t11[j].x, t11[j].y, t11[j].z, t11[j].w }, a01[4] = { t01[j].x, t01[j].y, t01[j].z, t01[j].w };
            float res[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) res[i] = attenuate_step<true>(axis0_blend(a00[i], a10[i], a11[i], a01[i], tp[j]), delta, n[i]);
            *reinterpret_cast<float4*>(dst + sy * (unsigned)(y - j)) = make_float4(res[0], res[1], res[2], res[3]);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) tp[j] = tn[j];
    }
    for (; s < steps; ++s, --y) {
        const RowTapsOff t = trow[y];
        const float4 b00 = tap4(src, t.o00, esz), b10 = tap4(src, t.o10, esz), b11 = tap4(src, t.o11, esz), b01 = tap4(src, t.o01, esz);
        const float a00[4] = { b00.x, b00.y, b00.z, b00.w }, a10[4] = { b10.x, b10.y, b10.z, b10.w };
        const float a11[4] = { b11.x, b11.y, b11.z, b11.w }, a01[4] = { b01.x, b01.y, b01.z, b01.w };
        float res[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) res[i] = attenuate_step<true>(axis0_blend(a00[i], a10[i], a11[i], a01[i], t), delta, n[i]);
        *reinterpret_cast<float4*>(dst + sy * (unsigned)y) = make_float4(res[0], res[1], res[2], res[3]);
    }
    for (; y >= 0; --y) *reinterpret_cast<float4*>(dst + sy * (unsigned)y) = make_float4(0.f, 0.f, 0.f, 0.f);
}

// a rotation about x: row 0 of the inverse is the identity (up to the rounding of (c^2+s^2) * 1/(c^2+s^2), < 1e-15), so x_src == x
// and the gather is bilinear in (y, z)
static bool x_identity(int axis, const double inv[12])
{
    return axis == 0 && fabs(inv[0] - 1.0) < 1e-12 && inv[1] == 0.0 && inv[2] == 0.0 && inv[3] == 0.0 && inv[4] == 0.0 && inv[8] == 0.0;
}

// returns MVSIM_EUNSUPPORTED when the fused path does not apply (caller falls back to the two kernels)
int k_rotate_attenuate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], int axis, const double inv[12], double delta, int steps,
                       int64_t z0, int64_t z_local)
{
    const int X = (int)dims[0], Y = (int)dims[1], Z = (int)dims[2];
    const int Zl = z_local > 0 ? (int)z_local : Z, zfirst = z_local > 0 ? (int)z0 : 0;
    if (!x_identity(axis, inv)) return MVSIM_EUNSUPPORTED;
    Affine a;
    for (int i = 0; i < 12; ++i) a.m[i] = inv[i];
    const bool aligned = (reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) % 16 == 0;
    // tabulated tap offsets (measured 0.857 -> 0.810 ms at config 3, profiles/r02h_rotate_ab.txt) wherever 32-bit offsets and float4 apply
    if (X % 4 == 0 && aligned && (double)X * Y * Z < 2147483648.0) {
        RowTapsOff* tabo = nullptr;
        MVSIM_TRY(dev_alloc(ctx, (void**)&tabo, sizeof(RowTapsOff) * (size_t)Y * Zl));
        rotate_rowtable_off_kernel<<<blocks_for((size_t)Y * Zl, 256), 256, 0, ctx->stream>>>(tabo, X, Y, Z, zfirst, Zl, a);
        ctx->launches++;
        // rows per batch: 3 -> 4 once the tap addresses were single instructions (62 -> 70 registers, still 7 CTAs of 128 threads per SM
        // = one wave at config 3): 0.798 -> 0.752 ms (profiles/r02_notes.md)
        // (CTAs of 64 threads: 0.738 against 0.740 ms -- no difference)
        rotate_attenuate_off_kernel<4><<<blocks_for((size_t)(X / 4) * Zl, 128), 128, 0, ctx->stream>>>(in, out, tabo, X, Y, delta, steps, Zl, (unsigned)sizeof(float));
        ctx->launches++;
        cudaError_t eo = cudaGetLastError();
        dev_free(ctx, tabo);
        if (eo != cudaSuccess) return cuda_fail(ctx, eo, "rotate_attenuate_off_kernel");
        return MVSIM_OK;
    }
    RowTaps* tab = nullptr;
    MVSIM_TRY(dev_alloc(ctx, (void**)&tab, sizeof(RowTaps) * (size_t)Y * Zl));
    rotate_rowtable_kernel<<<blocks_for((size_t)Y * Zl, 256), 256, 0, ctx->stream>>>(tab, Y, zfirst, Zl, a);
    ctx->launches++;
    // the march along y is sequential per column, so the grid is small (X*Z/VEC threads): the widest vector the row allows
    // (L2 prefetch of the source rows was measured and lost in both forms -- issued by thread 0: 0.905 -> 1.11 .. 1.31 ms; by a
    // fifth, paced warp per CTA: 1.04 .. 1.06 ms, profiles/r02_experiments.txt -- the march already keeps 2 rows x 4 taps in
    // flight per thread and re-reads every source row from the L2.)
    if (X % 4 == 0 && aligned) {
        const size_t cols = (size_t)(X / 4) * Zl;
        rotate_attenuate_kernel<4, 2><<<blocks_for(cols, 128), 128, 0, ctx->stream>>>(in, out, tab, X, Y, Z, delta, steps, Zl);
    } else if (X % 2 == 0 && aligned) {
        const size_t cols = (size_t)(X / 2) * Zl;
        rotate_attenuate_kernel<2, 4><<<blocks_for(cols, 128), 128, 0, ctx->stream>>>(in, out, tab, X, Y, Z, delta, steps, Zl);
    } else {
        const size_t cols = (size_t)X * Zl;
        rotate_attenuate_kernel<1, 4><<<blocks_for(cols, 128), 128, 0, ctx->stream>>>(in, out, tab, X, Y, Z, delta, steps, Zl);
    }
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    dev_free(ctx, tab);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "rotate_attenuate_kernel");
    return MVSIM_OK;
}

int k_rotate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], int axis, const double inv[12])
{
    Affine a;
    for (int i = 0; i < 12; ++i) a.m[i] = inv[i];
    const int X = (int)dims[0], Y = (int)dims[1], Z = (int)dims[2];
    if (x_identity(axis, inv)) {
        const bool vec4 = (X % 4 == 0) && ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) % 16 == 0);
        if (vec4) {
            const size_t total = (size_t)(X / 4) * Y * Z;
            rotate_axis0_kernel<4><<<blocks_for(total, 256), 256, 0, ctx->stream>>>(in, out, X, Y, Z, a);
        } else {
            const size_t total = (size_t)X * Y * Z;
            rotate_axis0_kernel<1><<<blocks_for(total, 256), 256, 0, ctx->stream>>>(in, out, X, Y, Z, a);
        }
    } else {
        const size_t total = (size_t)X * Y * Z;
        rotate_general_kernel<<<blocks_for(total, 256), 256, 0, ctx->stream>>>(in, out, X, Y, Z, a);
    }
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

// ---------------------------------------------------------------------------------------------
// attenuate.  One (x,z) column per thread (lanes along x: coalesced), marching from y = Y-1 down;
// the FP64 recurrence of :343-357 (attenuate_step: post.cuh).  The loads do not depend on the
// recurrence, so they are issued 8 rows ahead.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) attenuate_kernel(const float* __restrict__ in, float* __restrict__ out, int X, int Y, int Z,
                                                        double delta, int steps)
{
    const long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= (long long)X * Z) return;
    const int x = (int)(col % X), z = (int)(col / X);
    const long long base = x + (long long)X * Y * z;
    const float* p = in + base;
    float* o = out + base;
    double n = 1.0;
    int y = Y - 1, s = 0;
    for (; s + 8 <= steps; s += 8, y -= 8) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __ldg(p + (long long)(y - j) * X);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[(long long)(y - j) * X] = attenuate_step(v[j], delta, n);
    }
    for (; s < steps; ++s, --y) o[(long long)y * X] = attenuate_step(__ldg(p + (long long)y * X), delta, n);
    for (; y >= 0; --y) o[(long long)y * X] = 0.f;      // rows the reference loop never reaches stay 0 (:321)
}

int k_attenuate(mvsim_ctx* ctx, const float* in, float* out, const int64_t dims[3], double delta, int steps)
{
    const size_t cols = (size_t)dims[0] * dims[2];
    attenuate_kernel<<<blocks_for(cols, 128), 128, 0, ctx->stream>>>(in, out, (int)dims[0], (int)dims[1], (int)dims[2], delta, steps);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

// ---------------------------------------------------------------------------------------------
// deterministic double sums (RealSum replacement): fixed thread -> element assignment, fixed-order
// tree in shared memory, fixed-order second stage.  The result depends only on n.
// ---------------------------------------------------------------------------------------------
constexpr int kSumThreads = 256;
constexpr int kSumMaxBlocks = 1184;     // 8 CTAs per SM on 148 SMs

__device__ __forceinline__ double block_tree_sum(double v, double* sm)
{
    sm[threadIdx.x] = v;
    __syncthreads();
    for (int s = kSumThreads / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
        __syncthreads();
    }
    return sm[0];
}

__global__ void __launch_bounds__(kSumThreads) sum_stage1_kernel(const float* __restrict__ in, size_t n, double* __restrict__ partials)
{
    __shared__ double sm[kSumThreads];
    double acc = 0.0;
    const size_t stride = (size_t)gridDim.x * kSumThreads;
    for (size_t i = (size_t)blockIdx.x * kSumThreads + threadIdx.x; i < n; i += stride) acc += (double)__ldg(in + i);
    const double s = block_tree_sum(acc, sm);
    if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kSumThreads) sum_stage2_kernel(const double* __restrict__ partials, size_t n, double* __restrict__ out)
{
    __shared__ double sm[kSumThreads];
    double acc = 0.0;
    for (size_t i = threadIdx.x; i < n; i += kSumThreads) acc += partials[i];
    const double s = block_tree_sum(acc, sm);
    if (threadIdx.x == 0) *out = s;
}

int k_sum_partials(mvsim_ctx* ctx, const double* partials, size_t n, double* d_sum)
{
    sum_stage2_kernel<<<1, kSumThreads, 0, ctx->stream>>>(partials, n, d_sum);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

int k_sum(mvsim_ctx* ctx, const float* in, size_t n, double* d_sum)
{
    unsigned blocks = blocks_for(n, kSumThreads * 16);
    if (blocks > kSumMaxBlocks) blocks = kSumMaxBlocks;
    if (blocks < 1) blocks = 1;
    double* partials = nullptr;
    MVSIM_TRY(dev_alloc(ctx, (void**)&partials, sizeof(double) * blocks));
    sum_stage1_kernel<<<blocks, kSumThreads, 0, ctx->stream>>>(in, n, partials);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    int st = e == cudaSuccess ? k_sum_partials(ctx, partials, blocks, d_sum) : cuda_fail(ctx, e, "sum_stage1_kernel");
    dev_free(ctx, partials);
    return st;
}

// ---------------------------------------------------------------------------------------------
// 128-bit content hash for the PSF-spectrum cache: h_j = sum_i mix_j(bits_i, i) mod 2^64 for two independent finalisers
// (splitmix64 / murmur3 constants).  A sum is order independent, so the grid shape does not matter and integer atomics
// keep it deterministic.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long mix_a(unsigned long long z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ unsigned long long mix_b(unsigned long long z)
{
    z ^= z >> 33; z *= 0xFF51AFD7ED558CCDull;
    z ^= z >> 33; z *= 0xC4CEB9FE1A85EC53ull;
    return z ^ (z >> 33);
}

__global__ void __launch_bounds__(256) hash128_kernel(const float* __restrict__ in, size_t n, unsigned long long* __restrict__ out)
{
    unsigned long long a = 0, b = 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long w = ((unsigned long long)i << 32) ^ (unsigned long long)__float_as_uint(__ldg(in + i)) ^ ((unsigned long long)(i >> 32) * 0xD6E8FEB86659FD93ull);
        a += mix_a(w);
        b += mix_b(w ^ 0xA5A5A5A55A5A5A5Aull);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        a += __shfl_down_sync(0xffffffffu, a, d);
        b += __shfl_down_sync(0xffffffffu, b, d);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(out, a); atomicAdd(out + 1, b); }
}

int k_hash128(mvsim_ctx* ctx, const float* in, size_t n, unsigned long long* d_out)
{
    cudaError_t e = cudaMemsetAsync(d_out, 0, 2 * sizeof(unsigned long long), ctx->stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "hash memset");
    unsigned blocks = blocks_for(n, 256 * 8);
    if (blocks > 1184) blocks = 1184;
    if (blocks < 1) blocks = 1;
    hash128_kernel<<<blocks, 256, 0, ctx->stream>>>(in, n, d_out);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

// normImage: t = (float)((double)t / sum)   S/Tools.java:116-117
__global__ void __launch_bounds__(256) divide_by_sum_kernel(float* __restrict__ a, size_t n, const double* __restrict__ d_sum)
{
    const double sum = *d_sum;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = (float)((double)a[i] / sum);
}

int k_divide_by_sum(mvsim_ctx* ctx, float* inout, size_t n, const double* d_sum)
{
    divide_by_sum_kernel<<<blocks_for(n, 256), 256, 0, ctx->stream>>>(inout, n, d_sum);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

// adjustImage: correction = (targetAverage - minValue) / (sum / size)   S/Tools.java:146-147
__global__ void adjust_corr_kernel(const double* __restrict__ d_sum, double n, float min_value, float target_avg, double* __restrict__ d_corr)
{
    const double avg = *d_sum / n;
    *d_corr = (double)__fsub_rn(target_avg, min_value) / avg;
}

// correction from the per-rank sums of a slab-decomposed volume, added in rank order (the result does not depend on the collective's
// reduction order): avg = (sum_r s_r) / n_global
__global__ void adjust_corr_ranks_kernel(const double* __restrict__ d_sums, int world, double n, float min_value, float target_avg, double* __restrict__ d_corr)
{
    double s = 0.0;
    for (int r = 0; r < world; ++r) s += d_sums[r];
    *d_corr = (double)__fsub_rn(target_avg, min_value) / (s / n);
}

int k_adjust_corr_ranks(mvsim_ctx* ctx, const double* d_sums, int world, double n_global, float min_value, float target_avg, double* d_corr)
{
    adjust_corr_ranks_kernel<<<1, 1, 0, ctx->stream>>>(d_sums, world, n_global, min_value, target_avg, d_corr);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

int k_adjust_corr(mvsim_ctx* ctx, const double* d_sum, size_t n, float min_value, float target_avg, double* d_corr)
{
    adjust_corr_kernel<<<1, 1, 0, ctx->stream>>>(d_sum, (double)n, min_value, target_avg, d_corr);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

// t = (float)(t * correction); t = t + minValue   (two roundings, S/Tools.java:150-155)
__device__ __forceinline__ float adjust_one(float v, double corr, float min_value)
{
    return __fadd_rn((float)__dmul_rn((double)v, corr), min_value);
}

__global__ void __launch_bounds__(256) adjust_apply_kernel(float* __restrict__ a, size_t n, const double* __restrict__ d_corr, float min_value)
{
    const double corr = *d_corr;
    const size_t i4 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 + 4 <= n) {
        float4 v = *reinterpret_cast<float4*>(a + i4);
        v.x = adjust_one(v.x, corr, min_value); v.y = adjust_one(v.y, corr, min_value);
        v.z = adjust_one(v.z, corr, min_value); v.w = adjust_one(v.w, corr, min_value);
        *reinterpret_cast<float4*>(a + i4) = v;
    } else {
        for (size_t i = i4; i < n; ++i) a[i] = adjust_one(a[i], corr, min_value);
    }
}

int k_adjust_apply(mvsim_ctx* ctx, float* inout, size_t n, const double* d_corr, float min_value)
{
    if (reinterpret_cast<uintptr_t>(inout) % 16 != 0) return set_error(ctx, MVSIM_EINVAL, "adjust: buffer not 16-byte aligned");
    adjust_apply_kernel<<<blocks_for((n + 3) / 4, 256), 256, 0, ctx->stream>>>(inout, n, d_corr, min_value);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

// ---------------------------------------------------------------------------------------------
// extract + (adjust) + Poisson.  One output voxel per thread, x fastest; slice cz of the output is
// slice cz*inc of the input (:206, integer, bit exact).  lambda = v * mul, mul = (SNR/sqrt 5)^2
// (S/Tools.java:76); the output is the raw count (S/Tools.java:84).
// ---------------------------------------------------------------------------------------------
// Cooperative finish of the voxels whose first PTRS proposal was not accepted by the squeeze (about 20 % of the voxels with
// lambda >= 10).  Left to each thread, a warp would run the slow code up to four times with a handful of active lanes, so the
// pending voxels are compacted into shared memory and finished with (nearly) full warps.  History: per-warp lists of one group per
// thread ran the slow code with ~9 of 32 lanes; a CTA-wide list (64 threads, three __syncthreads) 0.93 ms on the profiling volume,
// 23 % of the stall samples at the barriers (ncu r02b); the kernel below -- per-warp lists of TWO groups per thread, the same list
// length without any block barrier -- 0.90 ms.  Re-compacting the survivors after every attempt was measured slower (1.39 ms).
// The result of a voxel depends on (seed, stream, voxel index) only.
struct PendingItem { double lam; unsigned long long index; uint32_t ru, rv; };

// One thread = G groups of four consecutive voxels (a warp owns 128 G consecutive voxels: float4 traffic when the plane size is a
// multiple of 4); the pending PTRS voxels of the WARP go to the warp's own shared-memory list (slots from a shared counter) and are
// finished with full warps -- no block barrier anywhere.
constexpr int kWarpSamplerThreads = 128;
template <int G> struct WarpSamplerShared {
    PendingItem items[32 * 4 * G];
    float results[32 * 4 * G];
    int count;
};

template <bool VEC4, int G> __global__ void __launch_bounds__(kWarpSamplerThreads) extract_warp_kernel(const float* __restrict__ in, float* __restrict__ out, long long plane,
                                                                          long long n_out, int inc, const double* __restrict__ d_corr,
                                                                          float min_value, int noise, double mul, PoissonKey key,
                                                                          long long in_plane0, long long group0,
                                                                          unsigned short* __restrict__ out16, int* __restrict__ overflow)
{
    __shared__ WarpSamplerShared<G> shw[kWarpSamplerThreads / 32];
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const long long gbase = ((long long)blockIdx.x * (kWarpSamplerThreads / 32) + w) * (32 * G);
    float v[G][4];
    bool valid[G];
    long long g[G];
#pragma unroll
    for (int k = 0; k < G; ++k) {
        g[k] = gbase + k * 32 + lane;
        const long long i0 = 4 * g[k];
        valid[k] = i0 < n_out;
#pragma unroll
        for (int j = 0; j < 4; ++j) v[k][j] = 0.f;
        if (valid[k]) {
            if (VEC4) {
                // inc == 1 (the whole-view call hands over the kept slices compacted): output voxel i reads input voxel
                // i + in_plane0 * plane -- no 64-bit division (a library call of ~60 instructions per group, ncu r02j)
                long long src_i = i0 + in_plane0 * plane;
                if (inc != 1) {
                    const long long cz = i0 / plane, r = i0 - cz * plane;
                    src_i = (cz * inc + in_plane0) * plane + r;
                }
                const float4 t = __ldg(reinterpret_cast<const float4*>(in + src_i));
                v[k][0] = t.x; v[k][1] = t.y; v[k][2] = t.z; v[k][3] = t.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const long long i = i0 + j < n_out ? i0 + j : n_out - 1;
                    const long long cz = i / plane, r = i - cz * plane;
                    v[k][j] = __ldg(in + (cz * inc + in_plane0) * plane + r);
                }
            }
        }
    }
    if (d_corr) {
        const double corr = *d_corr;
#pragma unroll
        for (int k = 0; k < G; ++k)
#pragma unroll
            for (int j = 0; j < 4; ++j) v[k][j] = adjust_one(v[k][j], corr, min_value);
    }
    if (noise) {
        // slots are handed out by a shared-memory counter as the pending voxels turn up (group by group, so nothing but the slot
        // numbers stays live in registers); a voxel's result depends on (seed, stream, voxel index) only, not on its slot
        WarpSamplerShared<G>& sh = shw[w];
        if (lane == 0) sh.count = 0;
        __syncwarp();
        unsigned long long slots[G];
#pragma unroll
        for (int k = 0; k < G; ++k) {
            double lam[4];
            Philox4 r0, r1;
#pragma unroll
            for (int j = 0; j < 4; ++j) lam[j] = valid[k] ? __dmul_rn((double)v[k][j], mul) : 0.0;
            const unsigned pending = poisson_group4_fast(lam, (uint64_t)(g[k] + group0), key, v[k], r0, r1);
            slots[k] = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (pending & (1u << j)) {
                    const int pos = atomicAdd(&sh.count, 1);
                    PendingItem it;
                    it.lam = lam[j];
                    it.index = 4ull * (unsigned long long)(g[k] + group0) + (unsigned)j;
                    it.ru = j == 0 ? r0.x : j == 1 ? r0.y : j == 2 ? r0.z : r0.w;
                    it.rv = j == 0 ? r1.x : j == 1 ? r1.y : j == 2 ? r1.z : r1.w;
                    sh.items[pos] = it;
                    slots[k] |= (unsigned long long)(pos + 1) << (16 * j);      // 0 = not pending
                }
        }
        __syncwarp();
        const int total = sh.count;
        if (total > 0) {                          // warp uniform
            for (int j = (int)lane; j < total; j += 32) {
                const PendingItem it = sh.items[j];
                sh.results[j] = ptrs_resolve(it.lam, it.ru, it.rv, it.index, key);
            }
            __syncwarp();
#pragma unroll
            for (int k = 0; k < G; ++k)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const unsigned sl = (unsigned)(slots[k] >> (16 * j)) & 0xffffu;
                    if (sl) v[k][j] = sh.results[sl - 1];
                }
        }
    }
#pragma unroll
    for (int k = 0; k < G; ++k) {
        if (!valid[k]) continue;
        const long long i0 = 4 * g[k];
        if (VEC4) {
            *reinterpret_cast<float4*>(out + i0) = make_float4(v[k][0], v[k][1], v[k][2], v[k][3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (i0 + j < n_out) out[i0 + j] = v[k][j];
        }
        if (out16) {
            bool over = false;
            unsigned short q[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                over |= !(v[k][j] <= 65535.0f);
                q[j] = (unsigned short)fminf(fmaxf(v[k][j], 0.f), 65535.0f);
            }
            if (VEC4) {
                *reinterpret_cast<ushort4*>(out16 + i0) = make_ushort4(q[0], q[1], q[2], q[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (i0 + j < n_out) out16[i0 + j] = q[j];
            }
            if (over) atomicOr(overflow, 1);
        }
    }
}

static double snr_to_mul(double snr) { const double q = snr / sqrt(5.0); return pow(q, 2.0); }

int k_extract(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, const double* d_corr, float min_value,
              float snr, uint64_t seed, uint64_t stream, float* out)
{
    return k_extract_slab(ctx, in, dims, 0, dims[2], inc, d_corr, min_value, snr, seed, stream, out, nullptr);
}

int k_extract_u16(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, const double* d_corr, float min_value,
                  float snr, uint64_t seed, uint64_t stream, float* out, unsigned short* out16, int* d_overflow)
{
    return k_extract_slab(ctx, in, dims, 0, dims[2], inc, d_corr, min_value, snr, seed, stream, out, nullptr, out16, d_overflow);
}

// extractSlices for the planes [z0, z0 + z_local) of a volume with global dims: keeps the global planes z % inc == 0 inside the
// slab, compacted in order (in = the slab, z_local planes).  z0 == 0 and z_local == dims[2]: the whole volume.
int k_extract_slab(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int64_t z0, int64_t z_local, int inc, const double* d_corr,
                   float min_value, float snr, uint64_t seed, uint64_t stream, float* out, int64_t* planes_out, unsigned short* out16,
                   int* d_overflow)
{
    const long long plane = (long long)dims[0] * dims[1];
    const long long k0 = (z0 + inc - 1) / inc;                                  // first kept plane index >= z0 / inc
    const long long k1 = (z0 + z_local - 1) / inc;                              // last kept plane index inside the slab
    const long long nz = (z_local > 0 && k1 >= k0 && k0 * inc < z0 + z_local) ? k1 - k0 + 1 : 0;
    if (planes_out) *planes_out = nz;
    if (nz == 0) return MVSIM_OK;
    const long long n_out = plane * nz;
    const int noise = snr >= 0.0f ? 1 : 0;
    const long long first = k0 * plane;                                         // global index of the slab's first output voxel
    if (first % 4 != 0) return set_error(ctx, MVSIM_EUNSUPPORTED, "extract (slab): X*Y*first_kept_plane must be a multiple of 4");
    const bool vec4 = plane % 4 == 0 && (reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) % 16 == 0;
    const double mul = snr_to_mul((double)snr);
    const PoissonKey key = make_poisson_key(seed, stream);
    const long long in_plane0 = k0 * inc - z0, group0 = first / 4;
    if (out16 && (reinterpret_cast<uintptr_t>(out16) % 8 != 0 || !d_overflow)) return set_error(ctx, MVSIM_EINVAL, "extract: uint16 buffer must be 8-byte aligned");
    const unsigned wblocks = blocks_for((size_t)((n_out + 3) / 4), (unsigned)(kWarpSamplerThreads * 2));
    if (vec4) extract_warp_kernel<true, 2><<<wblocks, kWarpSamplerThreads, 0, ctx->stream>>>(in, out, plane, n_out, inc, d_corr, min_value, noise, mul, key, in_plane0, group0, out16, d_overflow);
    else extract_warp_kernel<false, 2><<<wblocks, kWarpSamplerThreads, 0, ctx->stream>>>(in, out, plane, n_out, inc, d_corr, min_value, noise, mul, key, in_plane0, group0, out16, d_overflow);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

// ---------------------------------------------------------------------------------------------
// post-acquisition chain of main() (SURVEY section 8f-1)
//   makeIsotropic      S/SimulateMultiViewDataset.java:144-171   linear z up-sampling, mirror-single
//   computeWeightImage S/SimulateMultiViewDataset.java:280-316   cosine taper along y
//   weight normalisation                                 :615-661 the one cross-view reduction
// ---------------------------------------------------------------------------------------------
// x, y are integer positions, so the n-linear interpolation of :150,167 reduces to two taps along z (iso_plane, iso_blend: post.cuh)
__global__ void __launch_bounds__(256) make_isotropic_kernel(const float* __restrict__ in, float* __restrict__ out, long long plane, int Z,
                                                             long long n_out, int inc)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_out) return;
    const int zo = (int)(i / plane);
    const long long r = i - (long long)zo * plane;
    const IsoPlane p = iso_plane(zo, inc, Z);
    out[i] = iso_blend(__ldg(in + (long long)p.pa * plane + r), __ldg(in + (long long)p.pb * plane + r), p);
}

int k_make_isotropic(mvsim_ctx* ctx, const float* in, const int64_t dims[3], int inc, float* out)
{
    const long long plane = (long long)dims[0] * dims[1];
    const long long n_out = plane * ((dims[2] - 1) * inc + 1);
    make_isotropic_kernel<<<blocks_for((size_t)n_out, 256), 256, 0, ctx->stream>>>(in, out, plane, (int)dims[2], n_out, inc);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

__global__ void __launch_bounds__(256) weight_image_kernel(float* __restrict__ out, int X, int Y, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = weight_of_row((int)((i / X) % Y), Y);
}

int k_weight_image(mvsim_ctx* ctx, const int64_t dims[3], float* out)
{
    const size_t n = (size_t)dims[0] * dims[1] * dims[2];
    weight_image_kernel<<<blocks_for(n, 256), 256, 0, ctx->stream>>>(out, (int)dims[0], (int)dims[1], (long long)n);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

struct WeightPtrs { float* w[MVSIM_MAX_WEIGHT_VIEWS]; };

// float accumulation in view order like the cursors of :627-639; sum_out = sum of the normalised weights (:648-661)
__global__ void __launch_bounds__(256) normalize_weights_kernel(WeightPtrs p, int n_views, size_t n, float osem, float* __restrict__ sum_out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float v[MVSIM_MAX_WEIGHT_VIEWS];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < MVSIM_MAX_WEIGHT_VIEWS; ++k)
        if (k < n_views) { v[k] = p.w[k][i]; sum = __fadd_rn(sum, v[k]); }
    float s2 = 0.f;
#pragma unroll
    for (int k = 0; k < MVSIM_MAX_WEIGHT_VIEWS; ++k)
        if (k < n_views) {
            const float o = normalized_weight(v[k], sum, osem);
            p.w[k][i] = o;
            s2 = __fadd_rn(s2, o);
        }
    if (sum_out) sum_out[i] = s2;
}

int k_normalize_weights(mvsim_ctx* ctx, float* const* d_weights, int n_views, size_t n, float osem, float* d_sum_out)
{
    if (n_views < 1 || n_views > MVSIM_MAX_WEIGHT_VIEWS) return set_error(ctx, MVSIM_EINVAL, "normalize_weights: 1..%d views", MVSIM_MAX_WEIGHT_VIEWS);
    WeightPtrs p;
    for (int k = 0; k < MVSIM_MAX_WEIGHT_VIEWS; ++k) p.w[k] = k < n_views ? d_weights[k] : nullptr;
    normalize_weights_kernel<<<blocks_for(n, 256), 256, 0, ctx->stream>>>(p, n_views, n, osem, d_sum_out);
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

// ---------------------------------------------------------------------------------------------
// main()'s aligned outputs without the intermediate volumes (row / tap arithmetic: post.cuh)
//   align_view       rotateAroundAxis(makeIsotropic(acq, inc), 0, d)                    :588, :591
//   aligned_weights  normalised rotateAroundAxis(computeWeightImage(dims), 0, d_v)      :576, :592, :615-661
// Both launch 64 x 4 blocks: 64 threads along x, one output row (y, z) per warp pair, rows on grid x (no 64-bit division).
// ---------------------------------------------------------------------------------------------
template <int VEC> __device__ __forceinline__ bool any_negzero(const float (&a)[VEC])
{
    bool r = false;
#pragma unroll
    for (int i = 0; i < VEC; ++i) r |= __float_as_uint(a[i]) == 0x80000000u;
    return r;
}

template <int VEC> __device__ __forceinline__ void copy_vec(float (&d)[VEC], const float (&s)[VEC])
{
#pragma unroll
    for (int i = 0; i < VEC; ++i) d[i] = s[i];
}

// Values of the up-sampled volume at iso planes iz (p0, valid if z0) and iz+1 (p1, valid if z1) of one source row; rowp points at
// that row in acquired plane 0.  Each iso plane blends the acquired planes pa and pb.  The next iso plane lies between the same two
// planes or starts at pb, so two row loads serve both taps.  With w == 0 the blend f32(a + f32(b * 0)) equals a for finite b unless
// a is -0 (then the sign of b decides), so b is read only when it can change the result.
template <int VEC> __device__ __forceinline__ void iso_taps(const float* rowp, long long plane, bool z0, bool z1, const IsoPlane& p0,
                                                           const IsoPlane& p1, float (&v0)[VEC], float (&v1)[VEC])
{
    float a[VEC], b[VEC], a1[VEC], b1[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) { v0[i] = 0.f; v1[i] = 0.f; b[i] = 0.f; b1[i] = 0.f; }
    bool hb = false;
    if (z0) {
        vload<VEC>(a, rowp + p0.pa * plane, true);
        if (p0.w != 0.0 || any_negzero<VEC>(a)) { vload<VEC>(b, rowp + p0.pb * plane, true); hb = true; }
#pragma unroll
        for (int i = 0; i < VEC; ++i) v0[i] = iso_blend(a[i], b[i], p0);
    }
    if (z1) {
        if (z0 && p1.pa == p0.pa) copy_vec<VEC>(a1, a);
        else if (hb && p1.pa == p0.pb) copy_vec<VEC>(a1, b);
        else vload<VEC>(a1, rowp + p1.pa * plane, true);
        if (p1.w != 0.0 || any_negzero<VEC>(a1)) {
            if (hb && p1.pb == p0.pb) copy_vec<VEC>(b1, b);
            else vload<VEC>(b1, rowp + p1.pb * plane, true);
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) v1[i] = iso_blend(a1[i], b1[i], p1);
    }
}

// out: X x Y x Ziso, acq: X x Y x Za; tab: the rotation rows of the iso dims (rotate_rowtable_kernel)
template <int VEC> __global__ void __launch_bounds__(256) align_view_kernel(const float* __restrict__ acq, float* __restrict__ out,
                                                                           const RowTaps* __restrict__ tab, int X, int Y, int Ziso,
                                                                           int Za, int inc)
{
    const long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y;
    const int xv = blockIdx.y * blockDim.x + threadIdx.x;
    if (row >= (long long)Y * Ziso || xv * VEC >= X) return;
    const RowTaps t = tab[row];
    const long long plane = (long long)X * Y, x0 = (long long)xv * VEC;
    const bool y0 = (unsigned)t.iy < (unsigned)Y, y1 = (unsigned)(t.iy + 1) < (unsigned)Y;
    const bool z0 = (unsigned)t.iz < (unsigned)Ziso, z1 = (unsigned)(t.iz + 1) < (unsigned)Ziso;
    IsoPlane p0{}, p1{};
    if (z0) p0 = iso_plane(t.iz, inc, Za);
    if (z1) p1 = iso_plane(t.iz + 1, inc, Za);
    float a0[VEC], a1[VEC], b0[VEC], b1[VEC];          // a: source row iy (taps 00, 01), b: row iy + 1 (taps 10, 11)
    iso_taps<VEC>(acq + x0 + (long long)X * t.iy, plane, y0 && z0, y0 && z1, p0, p1, a0, a1);
    iso_taps<VEC>(acq + x0 + (long long)X * (t.iy + 1), plane, y1 && z0, y1 && z1, p0, p1, b0, b1);
    float r[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) r[i] = axis0_blend(a0[i], b0[i], b1[i], a1[i], t);
    *reinterpret_cast<typename VecT<VEC>::type*>(out + x0 + X * row) = *reinterpret_cast<typename VecT<VEC>::type*>(r);
}

int k_align_view(mvsim_ctx* ctx, const float* acq, const int64_t acq_dims[3], int inc, const double inv[12], float* out)
{
    const int X = (int)acq_dims[0], Y = (int)acq_dims[1], Za = (int)acq_dims[2];
    const int Ziso = (Za - 1) * inc + 1;
    Affine a;
    for (int i = 0; i < 12; ++i) a.m[i] = inv[i];
    const long long rows = (long long)Y * Ziso;
    RowTaps* tab = nullptr;
    MVSIM_TRY(dev_alloc(ctx, (void**)&tab, sizeof(RowTaps) * (size_t)rows));
    rotate_rowtable_kernel<<<blocks_for((size_t)rows, 256), 256, 0, ctx->stream>>>(tab, Y, 0, Ziso, a);
    ctx->launches++;
    const bool vec4 = X % 4 == 0 && (reinterpret_cast<uintptr_t>(acq) | reinterpret_cast<uintptr_t>(out)) % 16 == 0;
    const int xv = vec4 ? X / 4 : X;
    const dim3 block(64, 4), grid((unsigned)((rows + 3) / 4), (unsigned)((xv + 63) / 64));
    if (vec4) align_view_kernel<4><<<grid, block, 0, ctx->stream>>>(acq, out, tab, X, Y, Ziso, Za, inc);
    else align_view_kernel<1><<<grid, block, 0, ctx->stream>>>(acq, out, tab, X, Y, Ziso, Za, inc);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    dev_free(ctx, tab);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "align_view_kernel");
    return MVSIM_OK;
}

struct WeightViews { Affine a[MVSIM_MAX_WEIGHT_VIEWS]; int slot[MVSIM_MAX_WEIGHT_VIEWS]; };

// Row (y, z) of the Y x Z plane: the rotated-back weights of all n_all views, summed in view order and normalised exactly as
// normalize_weights_kernel does.  rows[slot * Y*Z + row] receives view k's normalised weight when wv.slot[k] >= 0, and
// rows[sum_slot * Y*Z + row] the sum of the normalised weights when sum_slot >= 0.
__global__ void __launch_bounds__(128) aligned_weight_rows_kernel(float* __restrict__ rows, int Y, int Z, int n_all, float osem, int sum_slot,
                                                                  WeightViews wv)
{
    const long long R = (long long)Y * Z;
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= R) return;
    const int y = (int)(row % Y), z = (int)(row / Y);
    float v[MVSIM_MAX_WEIGHT_VIEWS];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < MVSIM_MAX_WEIGHT_VIEWS; ++k)
        if (k < n_all) { v[k] = aligned_weight(y, z, Y, Z, wv.a[k]); sum = fadd_rn(sum, v[k]); }
    float s2 = 0.f;
#pragma unroll
    for (int k = 0; k < MVSIM_MAX_WEIGHT_VIEWS; ++k)
        if (k < n_all) {
            const float o = normalized_weight(v[k], sum, osem);
            s2 = fadd_rn(s2, o);
            if (wv.slot[k] >= 0) rows[wv.slot[k] * R + row] = o;
        }
    if (sum_slot >= 0) rows[sum_slot * R + row] = s2;
}

// out[x + X * row] = col[row]: a store-bound broadcast of one value per row
template <int VEC> __global__ void __launch_bounds__(256) broadcast_rows_kernel(const float* __restrict__ col, float* __restrict__ out, int X, long long R)
{
    const long long row = (long long)blockIdx.x * blockDim.y + threadIdx.y;
    const int xv = blockIdx.y * blockDim.x + threadIdx.x;
    if (row >= R || xv * VEC >= X) return;
    const float v = __ldg(col + row);
    float r[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) r[i] = v;
    *reinterpret_cast<typename VecT<VEC>::type*>(out + (long long)xv * VEC + X * row) = *reinterpret_cast<typename VecT<VEC>::type*>(r);
}

int k_aligned_weights(mvsim_ctx* ctx, const int64_t dims[3], int n_all, const double* inv, float osem, int n_out, const int* views,
                      float* const* outs, float* sum_out)
{
    const int X = (int)dims[0], Y = (int)dims[1], Z = (int)dims[2];
    const long long R = (long long)Y * Z;
    const int n_rows = n_out + (sum_out ? 1 : 0);
    if (n_rows == 0) return MVSIM_OK;
    WeightViews wv;
    for (int k = 0; k < MVSIM_MAX_WEIGHT_VIEWS; ++k) {
        wv.slot[k] = -1;
        for (int i = 0; i < 12; ++i) wv.a[k].m[i] = k < n_all ? inv[12 * k + i] : 0.0;
    }
    for (int j = 0; j < n_out; ++j) wv.slot[views[j]] = j;
    float* rows = nullptr;
    MVSIM_TRY(dev_alloc(ctx, (void**)&rows, sizeof(float) * (size_t)n_rows * (size_t)R));
    aligned_weight_rows_kernel<<<blocks_for((size_t)R, 128), 128, 0, ctx->stream>>>(rows, Y, Z, n_all, osem, sum_out ? n_out : -1, wv);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    for (int j = 0; j < n_rows && e == cudaSuccess; ++j) {
        float* dst = j < n_out ? outs[j] : sum_out;
        const bool vec4 = X % 4 == 0 && reinterpret_cast<uintptr_t>(dst) % 16 == 0;
        const int xv = vec4 ? X / 4 : X;
        const dim3 block(64, 4), grid((unsigned)((R + 3) / 4), (unsigned)((xv + 63) / 64));
        if (vec4) broadcast_rows_kernel<4><<<grid, block, 0, ctx->stream>>>(rows + (size_t)j * R, dst, X, R);
        else broadcast_rows_kernel<1><<<grid, block, 0, ctx->stream>>>(rows + (size_t)j * R, dst, X, R);
        ctx->launches++;
        e = cudaGetLastError();
    }
    dev_free(ctx, rows);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "aligned_weights");
    return MVSIM_OK;
}

__global__ void __launch_bounds__(256) poisson_kernel(float* __restrict__ a, size_t n, double mul, PoissonKey key)
{
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (4 * g >= n) return;
    double lam[4];
    float v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) lam[k] = 4 * g + k < n ? __dmul_rn((double)a[4 * g + k], mul) : 0.0;
    poisson_group4(lam, (uint64_t)g, key, v);
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (4 * g + k < n) a[4 * g + k] = v[k];
}

int k_poisson(mvsim_ctx* ctx, float* inout, size_t n, double snr, uint64_t seed, uint64_t stream)
{
    poisson_kernel<<<blocks_for((n + 3) / 4, 256), 256, 0, ctx->stream>>>(inout, n, snr_to_mul(snr), make_poisson_key(seed, stream));
    MVSIM_LAUNCH_CHECK(ctx);
    return MVSIM_OK;
}

}  // namespace mvsim
