// One-step lookahead (pcgrl_lookahead): for candidate j, the reward / done / changed / stats that pcgrl_step would
// return for env e = env_idx[j] if e took action j next -- with the env left exactly as it is.
//
// Incremental path, for shards with a search cache (binary, maps up to 16x16, one-cell actions): three launches and
// no grid copied.
//   k_la_act     thread per candidate: decode the action against e's grid / position / frozen mask (the step's
//                one_cell_action), done and changed from e's counters; a candidate that leaves the grid as it is gets
//                reward 0 and e's stats, the others are appended to the work list in `work` as (e, cell), and j beside it.
//   k_split_stats_inc<NW, TWO, true>  (step_split.cu) the step's incremental search from e's cache row, which it
//                only reads.  Candidates are ordered env-major by lookahead_all, so neighbouring claims share a row.
//   k_la_out     thread per listed candidate: fp64 loss(new) - loss(e's stats) under e's targets.
// The work-list header in `work` follows the step's protocol (worklist.cuh), so the three launches hand the list
// over without a sync and the next lookahead finds its counter cleared.
//
// Generic path, for every other config: k_la_gather copies each candidate's env rows into a sub-shard carved from
// `work`, and api.cu runs the ordinary MODE_STEP on it.
#include "pcgrl_device.cuh"
#include "step_common.cuh"
#include "worklist.cuh"

namespace pcgrl {

cudaError_t launch_lookahead_search(const KParams& p, cudaStream_t s);

constexpr int LA_THREADS = 256;

// candidate index of list item i, behind the item stats (the body is [(env, cell) | K stats | j] per item)
__device__ __forceinline__ int32_t* la_cand(const KParams& p) { return p.worklist + (2 + p.n_stats) * p.n_envs; }

template <int K>
__global__ void __launch_bounds__(LA_THREADS) k_la_act(const KParams p, const LaOut o) {
    const int64_t j = (int64_t)blockIdx.x * LA_THREADS + threadIdx.x;
    bool need = false;
    int cell = -1;
    int64_t e = 0;
    if (j < p.n_envs) {
        e = o.env_idx ? (int64_t)o.env_idx[j] : j;
        int32_t st[K];
        if ((uint64_t)e >= (uint64_t)o.n_src) {   // nothing is loaded through a bad index
            if (p.status) atomicOr(p.status, 128);
            o.reward[j] = 0.f;
            o.done[j] = 0;
            o.changed[j] = 0;
#pragma unroll
            for (int k = 0; k < K; ++k) st[k] = 0;
        } else {
            const int cw = one_cell_action<false>(p, j, e, &cell);
            const int change = cw & 1;
            o.done[j] = episode_done(p, p.iteration[e] + 1, p.changes[e] + change);
            o.changed[j] = change;
            need = (cw & 2) != 0;
#pragma unroll
            for (int k = 0; k < K; ++k) st[k] = p.stats[e * K + k];
            if (!need) o.reward[j] = 0.f;
        }
        if (!need)
#pragma unroll
            for (int k = 0; k < K; ++k) o.stats[j * K + k] = st[k];
    }
    const int slot = wl_append_slot<LA_THREADS>(p, need);
    if (need) {
        wl_items(p)[slot] = make_int2((int)e, cell);
        la_cand(p)[slot] = (int32_t)j;
    }
}

template <int K>
__global__ void __launch_bounds__(LA_THREADS) k_la_out(const KParams p, const LaOut o) {
    const int count = *(volatile const int*)(p.wl_hdr + 4);
    const int i = blockIdx.x * LA_THREADS + threadIdx.x;
    if (i == 0) p.wl_hdr[3] = p.wl_hdr[3] + 1;   // as k_split_out: the next lookahead uses the other counter
    if (i >= count) return;
    const int64_t e = wl_items(p)[i].x, j = la_cand(p)[i];
    int32_t nw[K], od[K];
    const int32_t* s = wl_stats(p) + (int64_t)i * K;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        nw[k] = s[k];
        od[k] = p.stats[e * K + k];
    }
    o.reward[j] = step_reward<K>(p, p.targets + (p.targets_per_env ? e * K * 2 : 0), nw, od);
#pragma unroll
    for (int k = 0; k < K; ++k) o.stats[j * K + k] = nw[k];
}

// Incremental path.  p: the shard's state (grids, pos, counters, stats, targets, static mask, cache) with n_envs =
// the candidate count, actions = the candidates', wl_hdr / worklist inside the caller's work buffer.
cudaError_t launch_lookahead_inc(const KParams& p, const LaOut& o, cudaStream_t s) {
    const unsigned blocks = (unsigned)((p.n_envs + LA_THREADS - 1) / LA_THREADS);
    k_la_act<2><<<blocks, LA_THREADS, 0, s>>>(p, o);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if ((e = launch_lookahead_search(p, s)) != cudaSuccess) return e;
    k_la_out<2><<<blocks, LA_THREADS, 0, s>>>(p, o);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Generic path: candidate j's rows of the shard `src` -> row j of the sub-shard `dst`.  One thread per 16-byte
// vector of the grid (and of the frozen mask); the thread of vector 0 also copies the small rows.  The old stats
// go straight into dst.stats, the caller's output, where the step reads and replaces them.
// ------------------------------------------------------------------------------------------------
struct LaGather {
    pcgrl_state src, dst;
    const int32_t* env_idx;
    int32_t chunks, K, hole_ints, targets_per_env;
};
__global__ void __launch_bounds__(LA_THREADS) k_la_gather(const LaGather g) {
    const int64_t i = (int64_t)blockIdx.x * LA_THREADS + threadIdx.x;
    const int64_t j = i / g.chunks;
    const int c = (int)(i - j * g.chunks);
    if (j >= g.dst.n_envs) return;
    const int64_t e = g.env_idx ? (int64_t)g.env_idx[j] : j;
    const bool ok = (uint64_t)e < (uint64_t)g.src.n_envs;   // a bad index loads nothing: its row is zeros
    const int64_t rs = (int64_t)g.chunks * 16;
    const uint4 z = make_uint4(0, 0, 0, 0);
    ((uint4*)(g.dst.grids + j * rs))[c] = ok ? ((const uint4*)(g.src.grids + e * rs))[c] : z;
    if (g.dst.static_mask)
        ((uint4*)(g.dst.static_mask + j * rs))[c] = ok ? ((const uint4*)(g.src.static_mask + e * rs))[c] : z;
    if (c) return;
    if (!ok && g.src.status) atomicOr(g.src.status, 128);
    for (int k = 0; k < 3; ++k) g.dst.pos[j * 3 + k] = ok ? g.src.pos[e * 3 + k] : 0;
    g.dst.n_step[j] = ok ? g.src.n_step[e] : 0;
    g.dst.iteration[j] = ok ? g.src.iteration[e] : 0;
    g.dst.changes[j] = ok ? g.src.changes[e] : 0;
    for (int k = 0; k < g.K; ++k) g.dst.stats[j * g.K + k] = ok ? g.src.stats[e * g.K + k] : 0;
    if (g.targets_per_env)
        for (int k = 0; k < 2 * g.K; ++k)
            ((double*)g.dst.targets)[j * 2 * g.K + k] = ok ? g.src.targets[e * 2 * g.K + k] : 0.0;
    if (g.dst.holes)
        for (int k = 0; k < g.hole_ints; ++k) g.dst.holes[j * g.hole_ints + k] = ok ? g.src.holes[e * g.hole_ints + k] : 0;
}

cudaError_t launch_lookahead_gather(const pcgrl_state& src, const pcgrl_state& dst, const int32_t* env_idx,
                                    int row_stride, int K, int hole_ints, bool targets_per_env, cudaStream_t s) {
    LaGather g;
    g.src = src;
    g.dst = dst;
    g.env_idx = env_idx;
    g.chunks = row_stride / 16;
    g.K = K;
    g.hole_ints = hole_ints;
    g.targets_per_env = targets_per_env;
    const int64_t threads = dst.n_envs * g.chunks;
    k_la_gather<<<(unsigned)((threads + LA_THREADS - 1) / LA_THREADS), LA_THREADS, 0, s>>>(g);
    return cudaGetLastError();
}

}  // namespace pcgrl
