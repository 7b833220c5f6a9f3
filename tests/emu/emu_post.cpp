// CPU evaluation of the row / tap arithmetic of the aligned outputs (multiview-simulation_b200/csrc/post.cuh is __host__ __device__):
// the same functions align_view_kernel and aligned_weight_rows_kernel call, looped over every voxel.
#include <stdint.h>

#include "post.cuh"

using namespace mvsim;

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
