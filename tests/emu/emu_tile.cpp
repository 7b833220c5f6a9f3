// CPU evaluation of the interval addressing of the sampler (multiview-simulation_b200/csrc/tile.cuh is __host__ __device__): the
// same make_tile_map / tile_group_offsets the interval instantiation of extract_warp_kernel calls.
#include <stdint.h>

#include "tile.cuh"

using namespace mvsim;

// parent offsets of the four voxels of each group starting at output index i0s[g] (a multiple of 4) -> off[4g .. 4g+3]
extern "C" void emu_tile_offsets(const int64_t dims[3], const int64_t min[3], const int64_t max[3], int inc, const uint64_t* i0s, long long n,
                                 long long* off)
{
    const TileMap m = make_tile_map(dims, min, max, inc);
    for (long long g = 0; g < n; ++g) {
        long long o[4];
        tile_group_offsets(m, i0s[g], o);
        for (int j = 0; j < 4; ++j) off[4 * g + j] = o[j];
    }
}
