// Row and tap arithmetic of the post-acquisition chain of main() (S/SimulateMultiViewDataset.java:576-663): the rotation rows of
// rotate_axis0_kernel, the z blend of makeIsotropic, the weight taper of computeWeightImage and the weight normalisation.
// __host__ __device__: the kernels in stages.cu and the CPU harness in tests/emu run this same code.  Every operation is an
// explicitly rounded IEEE operation (intrinsics on the device, plain operators on the host), so nothing is contracted into an FMA.
#pragma once
#include "fft/fft_defs.cuh"

namespace mvsim {

MVSIM_HD double dmul_rn(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
MVSIM_HD double dadd_rn(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
MVSIM_HD float fmul_rn(float a, float b)
{
#ifdef __CUDA_ARCH__
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
MVSIM_HD float fadd_rn(float a, float b)
{
#ifdef __CUDA_ARCH__
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
MVSIM_HD float fdiv_rn(float a, float b)
{
#ifdef __CUDA_ARCH__
    return __fdiv_rn(a, b);
#else
    return a / b;
#endif
}

// inverse affine of axisRotation (:80-102), 3x4 row-major
struct Affine { double m[12]; };

// One output row (y, z) of a rotation about x: the source rows (iy, iz) .. (iy+1, iz+1) and the bilinear weights
struct alignas(16) RowTaps { int iy, iz; float w00, w10, w11, w01; int pad0, pad1; };

// rotate_axis0_kernel's row arithmetic: x_src == x, so only l1*m(r,1) + l2*m(r,2) + m(r,3) of rows 1 and 2; floor and the
// fractional weights in FP64, the four products rounded to float; a far-outside coordinate is clamped before the int conversion
MVSIM_HD RowTaps axis0_row_taps(int y, int z, const Affine& a)
{
    const double ly = (double)y, lz = (double)z;
    const double py = dadd_rn(dadd_rn(dmul_rn(ly, a.m[5]), dmul_rn(lz, a.m[6])), a.m[7]);
    const double pz = dadd_rn(dadd_rn(dmul_rn(ly, a.m[9]), dmul_rn(lz, a.m[10])), a.m[11]);
    const double fy = floor(py), fz = floor(pz);
    const double wy = py - fy, wz = pz - fz;
    const double wyi = 1.0 - wy, wzi = 1.0 - wz;
    RowTaps t;
    t.iy = (int)fmax(fmin(fy, 2.0e9), -2.0e9);
    t.iz = (int)fmax(fmin(fz, 2.0e9), -2.0e9);
    t.w00 = (float)(wyi * wzi); t.w10 = (float)(wy * wzi); t.w11 = (float)(wy * wz); t.w01 = (float)(wyi * wz);
    t.pad0 = t.pad1 = 0;
    return t;
}

// imglib2's tap order 000, 100, 110, 010 reduced to (y, z): (iy, iz), (iy+1, iz), (iy+1, iz+1), (iy, iz+1)
MVSIM_HD float axis0_blend(float t00, float t10, float t11, float t01, const RowTaps& t)
{
    return fadd_rn(fadd_rn(fadd_rn(fmul_rn(t00, t.w00), fmul_rn(t10, t.w10)), fmul_rn(t11, t.w11)), fmul_rn(t01, t.w01));
}

// makeIsotropic (:144-171) at plane zo of the up-sampled volume: position (float)zo / (float)inc widened to double (:165), two taps
// along z over the mirror-single extension of the Za acquired planes
struct IsoPlane { int pa, pb; double wi, w; };

MVSIM_HD IsoPlane iso_plane(int zo, int inc, int Za)
{
    const double zf = (double)fdiv_rn((float)zo, (float)inc);
    const double f = floor(zf);
    IsoPlane p;
    p.w = zf - f;
    p.wi = 1.0 - p.w;
    const int iz = (int)f;
    p.pa = mirror_single(iz, Za);
    p.pb = mirror_single(iz + 1, Za);
    return p;
}

// f32(f32(a * (1 - w)) + f32(b * w))
MVSIM_HD float iso_blend(float a, float b, const IsoPlane& p)
{
    return fadd_rn((float)dmul_rn((double)a, p.wi), (float)dmul_rn((double)b, p.w));
}

// computeWeightImage (:280-316): cosine taper over the last 40 px of the lower half along y; constant along x and z
MVSIM_HD float weight_of_row(int y, int Y)
{
    const int l = Y - y - 1, half = Y / 2, span = 40;       // cosineSpan (:283)
    if (l < half) return 1.0f;
    if (l > half + span) return 0.0f;
    return (float)((cos(((double)(l - half) / (double)span) * 3.14159265358979323846) + 1.0) / 2.0);
}

// rotateAroundAxis(computeWeightImage(dims), 0, d) at row (y, z) of a Y x Z plane (:576, :592): the weight image is constant along
// x, so its rotation about x is too, and every tap reads the taper row it falls on (0 outside the volume)
MVSIM_HD float aligned_weight(int y, int z, int Y, int Z, const Affine& a)
{
    const RowTaps t = axis0_row_taps(y, z, a);
    const bool y0 = (unsigned)t.iy < (unsigned)Y, y1 = (unsigned)(t.iy + 1) < (unsigned)Y;
    const bool z0 = (unsigned)t.iz < (unsigned)Z, z1 = (unsigned)(t.iz + 1) < (unsigned)Z;
    const float w0 = y0 ? weight_of_row(t.iy, Y) : 0.f, w1 = y1 ? weight_of_row(t.iy + 1, Y) : 0.f;
    return axis0_blend(z0 ? w0 : 0.f, z0 ? w1 : 0.f, z1 ? w1 : 0.f, z1 ? w0 : 0.f, t);
}

// one view's normalised weight (:627-639): sum = float sum of all views' weights in view order
MVSIM_HD float normalized_weight(float v, float sum, float osem)
{
    return sum == 0.f ? 0.f : fminf(1.0f, fmul_rn(osem, fdiv_rn(v, sum)));
}

}  // namespace mvsim
