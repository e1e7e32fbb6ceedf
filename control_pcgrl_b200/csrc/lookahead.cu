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
// `work`, and api.cu runs the ordinary MODE_STEP on it.  pcgrl_step_envs takes the same path for shards without a work
// list, and k_step_envs_scatter writes the stepped rows back to their envs.
//
// With the observation (pcgrl_lookahead_obs) every candidate's after-state is a row of the sub-shard, and api.cu runs
// the unchanged observation writer on it.  The generic path leaves it there already; the incremental path runs
// k_la_gather before its three launches and k_la_apply (the step's apply_action on the copy) after them.
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
// Generic path (also pcgrl_step_envs' path for shards without a work list): row j of the sub-shard `sub` is env
// e = env_idx[j] (or j) of the shard `shard`.  One thread per 16-byte vector of the grid (and of the frozen mask); the
// thread of vector 0 also copies the small rows.
// k_la_gather: shard -> sub.  The old stats go to sub.stats (the lookahead's output, or step_envs' sub-shard), where
// the step reads and replaces them.  An index outside the shard loads nothing (its row is zeros) and sets status_bit.
// k_step_envs_scatter: sub -> shard, what the step wrote (grid, pos, counters, stats, reward, done, changed, record);
// an index outside the shard writes nothing.
// ------------------------------------------------------------------------------------------------
struct SubShard {
    pcgrl_state shard, sub;
    const int32_t* env_idx;
    int32_t chunks, K, hole_ints, targets_per_env, rec_ints, status_bit;
};
__global__ void __launch_bounds__(LA_THREADS) k_la_gather(const SubShard g) {
    const int64_t i = (int64_t)blockIdx.x * LA_THREADS + threadIdx.x;
    const int64_t j = i / g.chunks;
    const int c = (int)(i - j * g.chunks);
    if (j >= g.sub.n_envs) return;
    const int64_t e = g.env_idx ? (int64_t)g.env_idx[j] : j;
    const bool ok = (uint64_t)e < (uint64_t)g.shard.n_envs;   // a bad index loads nothing: its row is zeros
    const int64_t rs = (int64_t)g.chunks * 16;
    const uint4 z = make_uint4(0, 0, 0, 0);
    ((uint4*)(g.sub.grids + j * rs))[c] = ok ? ((const uint4*)(g.shard.grids + e * rs))[c] : z;
    if (g.sub.static_mask)
        ((uint4*)(g.sub.static_mask + j * rs))[c] = ok ? ((const uint4*)(g.shard.static_mask + e * rs))[c] : z;
    if (c) return;
    if (!ok && g.shard.status) atomicOr(g.shard.status, g.status_bit);
    for (int k = 0; k < 3; ++k) g.sub.pos[j * 3 + k] = ok ? g.shard.pos[e * 3 + k] : 0;
    g.sub.n_step[j] = ok ? g.shard.n_step[e] : 0;
    g.sub.iteration[j] = ok ? g.shard.iteration[e] : 0;
    g.sub.changes[j] = ok ? g.shard.changes[e] : 0;
    for (int k = 0; k < g.K; ++k) g.sub.stats[j * g.K + k] = ok ? g.shard.stats[e * g.K + k] : 0;
    if (g.targets_per_env)
        for (int k = 0; k < 2 * g.K; ++k)
            ((double*)g.sub.targets)[j * 2 * g.K + k] = ok ? g.shard.targets[e * 2 * g.K + k] : 0.0;
    if (g.sub.holes)
        for (int k = 0; k < g.hole_ints; ++k) g.sub.holes[j * g.hole_ints + k] = ok ? g.shard.holes[e * g.hole_ints + k] : 0;
    if (g.sub.records)   // the step leaves parts of the record as they were (the stats of an unchanged map)
        for (int k = 0; k < g.rec_ints; ++k)
            ((int32_t*)g.sub.records)[j * g.rec_ints + k] = ok ? ((const int32_t*)g.shard.records)[e * g.rec_ints + k] : 0;
}

__global__ void __launch_bounds__(LA_THREADS) k_step_envs_scatter(const SubShard g) {
    const int64_t i = (int64_t)blockIdx.x * LA_THREADS + threadIdx.x;
    const int64_t j = i / g.chunks;
    const int c = (int)(i - j * g.chunks);
    if (j >= g.sub.n_envs) return;
    const int64_t e = g.env_idx[j];
    if ((uint64_t)e >= (uint64_t)g.shard.n_envs) return;   // the gather set the status bit
    const int64_t rs = (int64_t)g.chunks * 16;
    ((uint4*)(g.shard.grids + e * rs))[c] = ((const uint4*)(g.sub.grids + j * rs))[c];
    if (c) return;
    for (int k = 0; k < 3; ++k) g.shard.pos[e * 3 + k] = g.sub.pos[j * 3 + k];
    g.shard.n_step[e] = g.sub.n_step[j];
    g.shard.iteration[e] = g.sub.iteration[j];
    g.shard.changes[e] = g.sub.changes[j];
    for (int k = 0; k < g.K; ++k) g.shard.stats[e * g.K + k] = g.sub.stats[j * g.K + k];
    g.shard.reward[e] = g.sub.reward[j];
    g.shard.done[e] = g.sub.done[j];
    if (g.shard.changed) g.shard.changed[e] = g.sub.changed[j];
    if (g.sub.records)
        for (int k = 0; k < g.rec_ints; ++k)
            ((int32_t*)g.shard.records)[e * g.rec_ints + k] = ((const int32_t*)g.sub.records)[j * g.rec_ints + k];
}

static SubShard sub_shard(const pcgrl_state& shard, const pcgrl_state& sub, const int32_t* env_idx, int row_stride,
                          int K, int hole_ints, bool targets_per_env, int rec_stride, int status_bit) {
    SubShard g;
    g.shard = shard;
    g.sub = sub;
    g.env_idx = env_idx;
    g.chunks = row_stride / 16;
    g.K = K;
    g.hole_ints = hole_ints;
    g.targets_per_env = targets_per_env;
    g.rec_ints = rec_stride / 4;
    g.status_bit = status_bit;
    return g;
}
static unsigned sub_blocks(const SubShard& g) {
    return (unsigned)((g.sub.n_envs * g.chunks + LA_THREADS - 1) / LA_THREADS);
}

cudaError_t launch_lookahead_gather(const pcgrl_state& shard, const pcgrl_state& sub, const int32_t* env_idx,
                                    int row_stride, int K, int hole_ints, bool targets_per_env, int rec_stride,
                                    int status_bit, cudaStream_t s) {
    const SubShard g = sub_shard(shard, sub, env_idx, row_stride, K, hole_ints, targets_per_env, rec_stride, status_bit);
    k_la_gather<<<sub_blocks(g), LA_THREADS, 0, s>>>(g);
    return cudaGetLastError();
}

cudaError_t launch_step_envs_scatter(const pcgrl_state& shard, const pcgrl_state& sub, const int32_t* env_idx,
                                     int row_stride, int K, int rec_stride, cudaStream_t s) {
    const SubShard g = sub_shard(shard, sub, env_idx, row_stride, K, 0, false, rec_stride, 0);
    k_step_envs_scatter<<<sub_blocks(g), LA_THREADS, 0, s>>>(g);
    return cudaGetLastError();
}

// pcgrl_lookahead_obs on a shard with a search cache: the incremental lookahead gives the outputs but no grid, so
// k_la_gather copies e's rows into the sub-shard and this kernel, a thread per candidate, applies the candidate's edit
// and position advance to row j of the copy with the step's own decode (apply_action).  p: the sub-shard (n_envs =
// the candidate count), actions = the candidates'.  A row gathered through a bad index stays as the gather left it.
__global__ void __launch_bounds__(LA_THREADS) k_la_apply(const KParams p, const int32_t* env_idx, int64_t n_src) {
    const int64_t j = (int64_t)blockIdx.x * LA_THREADS + threadIdx.x;
    if (j >= p.n_envs) return;
    if (env_idx && (uint64_t)env_idx[j] >= (uint64_t)n_src) return;
    apply_action(p, j);
}

cudaError_t launch_lookahead_apply(const KParams& p, const int32_t* env_idx, int64_t n_src, cudaStream_t s) {
    k_la_apply<<<(unsigned)((p.n_envs + LA_THREADS - 1) / LA_THREADS), LA_THREADS, 0, s>>>(p, env_idx, n_src);
    return cudaGetLastError();
}

}  // namespace pcgrl
