// Row and tap arithmetic of the rotation about x and of the attenuation (S/SimulateMultiViewDataset.java:104-135, :318-364) and of
// the post-acquisition chain of main() (:576-663): the rotation rows and their blend, the attenuation recurrence, the z blend of
// makeIsotropic, the weight taper of computeWeightImage and the weight normalisation.  Every kernel that rotates about x or
// attenuates calls these functions, so their results agree bit for bit.
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
MVSIM_HD double dsub_rn(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
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

// The row taps of an X x Y x Z volume (< 2^31 voxels) as element offsets from the row's x: the source rows (iy, iz), (iy+1, iz),
// (iy+1, iz+1), (iy, iz+1).  A tap outside the volume gets weight 0 and the offset of row (0, 0), so a march reads all four rows
// without a bounds test.  Its product f32(s * 0) with the voxel s of row (0, 0) is +0, like the product of the zero a bounds test
// substitutes, whenever s is finite and neither negative nor -0.  So for finite source data without negative values, which every
// generator here produces, the blend is bit-identical to the bounds-tested one.  For other finite data only the sign of a zero can
// differ: with all four taps outside and a negative voxel in row (0, 0) the blend is -0 where the bounds test gives +0.
struct alignas(16) RowTapsOff { unsigned o00, o10, o11, o01; float w00, w10, w11, w01; };

MVSIM_HD RowTapsOff axis0_row_offsets(const RowTaps& t, int X, int Y, int Z)
{
    const bool y0 = (unsigned)t.iy < (unsigned)Y, y1 = (unsigned)(t.iy + 1) < (unsigned)Y;
    const bool z0 = (unsigned)t.iz < (unsigned)Z, z1 = (unsigned)(t.iz + 1) < (unsigned)Z;
    const unsigned sy = (unsigned)X, sz = (unsigned)X * (unsigned)Y;
    RowTapsOff o;
    o.o00 = (y0 && z0) ? sy * (unsigned)t.iy + sz * (unsigned)t.iz : 0u;
    o.o10 = (y1 && z0) ? sy * (unsigned)(t.iy + 1) + sz * (unsigned)t.iz : 0u;
    o.o11 = (y1 && z1) ? sy * (unsigned)(t.iy + 1) + sz * (unsigned)(t.iz + 1) : 0u;
    o.o01 = (y0 && z1) ? sy * (unsigned)t.iy + sz * (unsigned)(t.iz + 1) : 0u;
    o.w00 = (y0 && z0) ? t.w00 : 0.f;
    o.w10 = (y1 && z0) ? t.w10 : 0.f;
    o.w11 = (y1 && z1) ? t.w11 : 0.f;
    o.w01 = (y0 && z1) ? t.w01 : 0.f;
    return o;
}

// imglib2's tap order 000, 100, 110, 010 reduced to (y, z): (iy, iz), (iy+1, iz), (iy+1, iz+1), (iy, iz+1); Taps: RowTaps or RowTapsOff
template <class Taps> MVSIM_HD float axis0_blend(float t00, float t10, float t11, float t01, const Taps& t)
{
    return fadd_rn(fadd_rn(fadd_rn(fmul_rn(t00, t.w00), fmul_rn(t10, t.w10)), fmul_rn(t11, t.w11)), fmul_rn(t01, t.w01));
}

// Math.max(d, 0) of :354 for a non-NaN d through the sign bit (one compare + two selects instead of the four instructions of a
// double-precision fmax on the device); -0.0 gives +0.0 like Math.max
MVSIM_HD double clamp0(double d)
{
#ifdef __CUDA_ARCH__
    return __double2hiint(d) < 0 ? 0.0 : d;
#else
    return signbit(d) ? 0.0 : d;
#endif
}

// One row of attenuate's recurrence (:343-357) with n the light left in the column: phi = v * delta * n, n = max(n - phi, 0),
// result f32(v * n).  SIGN_CLAMP takes the max through clamp0, which equals fmax for every non-NaN difference.
template <bool SIGN_CLAMP = false> MVSIM_HD float attenuate_step(float v, double delta, double& n)
{
    const double dv = (double)v;
    const double phi = dmul_rn(dmul_rn(dv, delta), n);
    const double d = dsub_rn(n, phi);
    n = SIGN_CLAMP ? clamp0(d) : fmax(d, 0.0);
    return (float)dmul_rn(dv, n);
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
