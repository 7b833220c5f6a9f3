// CPU evaluation of the row / tap arithmetic of the rotation about x, the attenuation and the aligned outputs
// (multiview-simulation_b200/csrc/post.cuh is __host__ __device__): the same functions the kernels in stages.cu call, looped over
// every voxel.
#include <stdint.h>

#include "post.cuh"

using namespace mvsim;

// rotateAroundAxis(in, 0, .) of an X x Y x Z volume with the bounds-tested taps of rotate_axis0_kernel
extern "C" void emu_rotate_axis0(const float* in, int X, int Y, int Z, const double inv[12], float* out)
{
    Affine a;
    for (int i = 0; i < 12; ++i) a.m[i] = inv[i];
    auto at = [&](int x, int yy, int zz) -> float {
        if ((unsigned)yy >= (unsigned)Y || (unsigned)zz >= (unsigned)Z) return 0.f;
        return in[x + X * (yy + (long long)Y * zz)];
    };
    for (int z = 0; z < Z; ++z)
        for (int y = 0; y < Y; ++y) {
            const RowTaps t = axis0_row_taps(y, z, a);
            for (int x = 0; x < X; ++x)
                out[x + X * (y + (long long)Y * z)] = axis0_blend(at(x, t.iy, t.iz), at(x, t.iy + 1, t.iz), at(x, t.iy + 1, t.iz + 1),
                                                                  at(x, t.iy, t.iz + 1), t);
        }
}

// rotate_attenuate_off_kernel: every (x, z) column marched from y = Y-1 down over the offset table, `steps` rows of the
// recurrence, the rows below stay 0
extern "C" void emu_rotate_attenuate_off(const float* in, int X, int Y, int Z, const double inv[12], double delta, int steps, float* out)
{
    Affine a;
    for (int i = 0; i < 12; ++i) a.m[i] = inv[i];
    for (int z = 0; z < Z; ++z)
        for (int x = 0; x < X; ++x) {
            const float* src = in + x;
            double n = 1.0;
            for (int y = Y - 1, s = 0; y >= 0; --y, ++s) {
                float r = 0.f;
                if (s < steps) {
                    const RowTapsOff t = axis0_row_offsets(axis0_row_taps(y, z, a), X, Y, Z);
                    r = attenuate_step<true>(axis0_blend(src[t.o00], src[t.o10], src[t.o11], src[t.o01], t), delta, n);
                }
                out[x + X * (y + (long long)Y * z)] = r;
            }
        }
}

// rotateAroundAxis(makeIsotropic(acq, inc), 0, .) of an X x Y x Za volume; inv = the axis-0 inverse of the isotropic dims
extern "C" void emu_align_view(const float* acq, int X, int Y, int Za, int inc, const double inv[12], float* out)
{
    Affine a;
    for (int i = 0; i < 12; ++i) a.m[i] = inv[i];
    const int Ziso = (Za - 1) * inc + 1;
    const long long plane = (long long)X * Y;
    auto iso = [&](int x, int yy, int zz) -> float {
        if ((unsigned)yy >= (unsigned)Y || (unsigned)zz >= (unsigned)Ziso) return 0.f;
        const IsoPlane p = iso_plane(zz, inc, Za);
        const long long r = x + (long long)X * yy;
        return iso_blend(acq[p.pa * plane + r], acq[p.pb * plane + r], p);
    };
    for (int z = 0; z < Ziso; ++z)
        for (int y = 0; y < Y; ++y) {
            const RowTaps t = axis0_row_taps(y, z, a);
            for (int x = 0; x < X; ++x)
                out[x + X * (y + (long long)Y * z)] = axis0_blend(iso(x, t.iy, t.iz), iso(x, t.iy + 1, t.iz), iso(x, t.iy + 1, t.iz + 1),
                                                                  iso(x, t.iy, t.iz + 1), t);
        }
}

// the normalised rotate-back weights of n_all views (inv: n_all x 12) over X x Y x Z: out[k] for every view, sum (nullable)
extern "C" void emu_aligned_weights(int X, int Y, int Z, int n_all, const double* inv, float osem, float* const* out, float* sum)
{
    for (int z = 0; z < Z; ++z)
        for (int y = 0; y < Y; ++y) {
            float v[64], s = 0.f, s2 = 0.f;
            for (int k = 0; k < n_all; ++k) {
                Affine a;
                for (int i = 0; i < 12; ++i) a.m[i] = inv[12 * k + i];
                v[k] = aligned_weight(y, z, Y, Z, a);
                s = fadd_rn(s, v[k]);
            }
            for (int k = 0; k < n_all; ++k) {
                const float o = normalized_weight(v[k], s, osem);
                s2 = fadd_rn(s2, o);
                for (int x = 0; x < X; ++x) out[k][x + X * (y + (long long)Y * z)] = o;
            }
            if (sum)
                for (int x = 0; x < X; ++x) sum[x + X * (y + (long long)Y * z)] = s2;
        }
}
