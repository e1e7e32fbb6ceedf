// What api.cu needs from level_distance.cu: the packed-level geometry, the work-buffer layout and the launches.
// The layout is decided in level_distance.cu alone; api.cu checks the arguments and calls these.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pcgrl {

// A level is `cells` tile codes; packed, it is W = ceil(cells / 32) words of each of P = ceil(log2 n_tiles) bit-planes
// (at least one), L = W * P words, word-major.
struct LdGeom {
    int cells, W, P, L;
};
LdGeom ld_geom(int cells, int n_tiles);
// false: a level of this size does not fit the distance tile's shared memory (PCGRL_E_UNSUPPORTED)
bool ld_fits(const LdGeom& g);
// Bytes of work for n_a packed levels, n_b packed levels and, for k > 0, the partial kNN lists of the split.
int64_t ld_work_bytes(const LdGeom& g, int64_t n_a, int64_t n_b, int k);

// `n` levels of `stride` bytes from `p` (device); only the first g.cells bytes of each are read.
struct LdLevels {
    const uint8_t* p;
    int64_t n, stride;
};
// Each returns the first CUDA error and adds the kernels it launched to n_launches.
cudaError_t launch_level_distances(const LdGeom& g, const LdLevels& a, const LdLevels& b, int32_t* out, void* work,
                                   cudaStream_t s, int& n_launches);
cudaError_t launch_level_knn(const LdGeom& g, const LdLevels& q, const LdLevels& b, int k, int64_t self_offset,
                             int32_t* dist, int32_t* idx, void* work, cudaStream_t s, int& n_launches);
cudaError_t launch_level_groups(const LdGeom& g, const LdLevels& a, int64_t group_size, int64_t* sums, void* work,
                                cudaStream_t s, int& n_launches);

}  // namespace pcgrl
