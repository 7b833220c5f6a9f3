// Output index -> parent offset of extractSlices (S/SimulateMultiViewDataset.java:195-231) over an interval of a larger volume,
// i.e. of Views.zeroMin(Views.interval(parent, min, max)) (S/SimulateTileStitching.java:152-153,174) without materialising the view.
// Output voxel (x, y, k) of the (bx, by, (bz-1)/inc+1) tile, b = max - min + 1, is parent voxel (min0 + x, min1 + y, min2 + k*inc).
// __host__ __device__: extract_warp_kernel in stages.cu and the CPU harness in tests/emu run this same code.
#pragma once
#include <stdint.h>

#include "fft/fft_defs.cuh"
#include "sampler.cuh"

namespace mvsim {

MVSIM_HD uint64_t mulhi64(uint64_t a, uint64_t b)
{
#ifdef __CUDA_ARCH__
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// The parent is addressed with 64 bits; the tile plane bx*by must fit in 32 bits (make_tile_map's caller checks it).
struct TileMap {
    long long base;          // parent offset of (min0, min1, min2)
    long long row_skip;      // parent X - bx: from the end of a tile row to the start of the next
    long long plane_skip;    // parent X*Y*inc - by*X: from the end of a kept tile plane to the start of the next
    long long row;           // parent X
    long long kept_plane;    // parent X*Y*inc
    uint64_t plane_magic;    // floor((2^64 - 1) / tile_plane)
    uint32_t bx, by, tile_plane;
    uint32_t row_magic;      // floor((2^32 - 1) / bx)
};

inline TileMap make_tile_map(const int64_t dims[3], const int64_t min[3], const int64_t max[3], int inc)
{
    TileMap m;
    m.bx = (uint32_t)(max[0] - min[0] + 1);
    m.by = (uint32_t)(max[1] - min[1] + 1);
    m.tile_plane = m.bx * m.by;
    m.row = dims[0];
    m.kept_plane = (long long)dims[0] * dims[1] * inc;
    m.base = min[0] + dims[0] * (min[1] + dims[1] * min[2]);
    m.row_skip = m.row - m.bx;
    m.plane_skip = m.kept_plane - (long long)m.by * m.row;
    m.plane_magic = UINT64_MAX / m.tile_plane;
    m.row_magic = UINT32_MAX / m.bx;
    return m;
}

// Parent offsets of the four output voxels i0 .. i0+3 (i0 = 4g, the sampler's Philox group g).  A group may straddle two rows or
// two kept planes.  The quotients come from high products with floor((2^N - 1) / d), which are the exact quotient or one less,
// and one correction step: no 64-bit division (a library call of ~60 instructions per group, ncu r02j).  Offsets of voxels
// at or past the tile's end are not inside the tile and must not be read.
MVSIM_HD void tile_group_offsets(const TileMap& m, uint64_t i0, long long (&off)[4])
{
    uint64_t k = mulhi64(i0, m.plane_magic);
    uint64_t r = i0 - k * m.tile_plane;
    if (r >= m.tile_plane) { ++k; r -= m.tile_plane; }
    uint32_t y = mulhi32((uint32_t)r, m.row_magic);
    uint32_t x = (uint32_t)r - y * m.bx;
    if (x >= m.bx) { ++y; x -= m.bx; }
    long long o = m.base + (long long)k * m.kept_plane + (long long)y * m.row + x;
    off[0] = o;
    MVSIM_UNROLL
    for (int j = 1; j < 4; ++j) {
        ++o;
        if (++x == m.bx) {
            x = 0;
            o += m.row_skip;
            if (++y == m.by) { y = 0; o += m.plane_skip; }
        }
        off[j] = o;
    }
}

}  // namespace mvsim
