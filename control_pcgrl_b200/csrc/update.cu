// Representation.update without get_stats (pcgrl_update): what evolution's generator loop calls at every iteration
// (evo/evolve.py:1082-1085, env built with _get_stats_on_step = False).  One launch edits the maps, advances pos /
// n_step and writes changed[N]; it never reads or writes iteration, changes, stats, reward, done, records or the
// split path's work list and search cache.
//
// The edit itself is the step kernels' own code (step_common.cuh): apply_action for the narrow / turtle / wide / patch
// representations, cellular_rewrite for the cellular one, so update and step cannot drift apart.
#include <algorithm>

#include "step_common.cuh"

namespace pcgrl {

constexpr int UPD_THREADS = 256;
constexpr int UPD_TILE = 256;   // most envs per CTA trip of the cellular rewrite

// CELLULAR: the whole-map rewrite over CTA tiles of `tile` (<= UPD_TILE) envs; else one thread per env.  (One body
// for both made ptxas keep the cellular loop counter in local memory.)
template <bool CELLULAR>
__global__ void __launch_bounds__(UPD_THREADS) k_update(const KParams p, const int tile) {
    const int tid = threadIdx.x;
    if constexpr (CELLULAR) {
        __shared__ uint8_t s_flag[UPD_TILE];
        for (int64_t base = (int64_t)blockIdx.x * tile; base < p.n_envs; base += (int64_t)gridDim.x * tile) {
            const int tile_n = (int)min((int64_t)tile, p.n_envs - base);
            for (int e = tid; e < UPD_TILE; e += UPD_THREADS) s_flag[e] = 0;
            __syncthreads();
            cellular_rewrite<UPD_THREADS>(p, base, tile_n, s_flag);
            // a thread reads back exactly the flags it zeroes on the next trip, so no barrier is needed in between
            for (int e = tid; e < tile_n; e += UPD_THREADS) p.changed[base + e] = s_flag[e];
        }
    } else {
        // bit0 of apply_action is the reference's `change`: under StaticTileRepresentation an undone edit of a frozen
        // cell still counts (step_common.cuh, apply_action)
        const int64_t stride = (int64_t)gridDim.x * UPD_THREADS;
        for (int64_t gid = (int64_t)blockIdx.x * UPD_THREADS + tid; gid < p.n_envs; gid += stride)
            p.changed[gid] = (uint8_t)(apply_action(p, gid) & 1);
    }
}

// Persistent grid: as many CTAs as are resident at once, or fewer when the shard is smaller.
cudaError_t launch_update(const KParams& p, cudaStream_t s) {
    static int per_sm[2] = {0, 0};
    int n_sm = 0;
    cudaError_t e;
    if ((e = sm_count(n_sm)) != cudaSuccess) return e;
    if (!per_sm[0] &&
        ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[0], k_update<false>, UPD_THREADS, 0)) != cudaSuccess ||
         (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[1], k_update<true>, UPD_THREADS, 0)) != cudaSuccess))
        return e;
    if (p.n_envs == 0) return cudaSuccess;
    const bool ca = p.rep == PCGRL_REP_CELLULAR;
    const int64_t cap = (int64_t)n_sm * (per_sm[ca] > 0 ? per_sm[ca] : 1);
    // cellular: envs per CTA trip so that one wave of CTAs covers the shard, at most UPD_TILE -- with whole tiles of
    // UPD_TILE envs a shard of large maps (smb 116x16, 64 Ki envs: 256 tiles) leaves most SMs without work
    const int64_t tile = ca ? std::min<int64_t>(std::max<int64_t>((p.n_envs + cap - 1) / cap, 1), UPD_TILE) : UPD_THREADS;
    const int64_t want = (p.n_envs + tile - 1) / tile;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    if (ca) k_update<true><<<grid, UPD_THREADS, 0, s>>>(p, (int)tile);
    else k_update<false><<<grid, UPD_THREADS, 0, s>>>(p, (int)tile);
    return cudaGetLastError();
}

}  // namespace pcgrl
