// The global work list of the split step path (step_split.cu) and of the incremental lookahead (lookahead.cu):
// envs whose map changed, appended by a thread-per-env kernel, searched by a second kernel and finished by a third.
#pragma once
#include "pcgrl_device.cuh"

namespace pcgrl {

// Work list of one launch: p.wl_hdr = 16 header ints, p.worklist = the body: (env, cell) pairs for up to n_envs items, then n_stats new
// stats per item.  The headers of all pipeline chunks live together at the front of pcgrl_state.worklist, where no
// body ever lands, so they stay zero whatever chunking the previous step used.
// Header (all zero before the first step): [0], [1] item counters used alternately, [3] the step count, whose parity
// picks the counter, [4] the step's final item count.  k_split_act adds to counter [par]; the search kernel clears
// counter [par ^ 1] for the next step and publishes the count in [4]; k_split_out reads [4] and bumps [3] -- every
// word is written by exactly one thread of a kernel none of whose CTAs reads it, so the three launches need no
// "last CTA out" atomics or fences to hand the list over.
__device__ __forceinline__ int wl_parity(const KParams& p) { return *(volatile const int*)(p.wl_hdr + 3) & 1; }
__device__ __forceinline__ int wl_count_search(const KParams& p) {
    const int par = wl_parity(p);
    const int count = *(volatile const int*)(p.wl_hdr + par);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        p.wl_hdr[par ^ 1] = 0;
        p.wl_hdr[4] = count;
    }
    return count;
}
__device__ __forceinline__ int2* wl_items(const KParams& p) { return (int2*)p.worklist; }
__device__ __forceinline__ int32_t* wl_stats(const KParams& p) { return p.worklist + 2 * p.n_envs; }

// CTA-aggregated append to the work list (one atomic per CTA): every thread of the CTA calls this; returns the list
// slot of this thread's item when `need`.
template <int THREADS>
__device__ __forceinline__ int wl_append_slot(const KParams& p, bool need) {
    __shared__ int s_warp[THREADS / 32];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned bal = __ballot_sync(0xffffffffu, need);
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) {
            const int c = s_warp[w];
            s_warp[w] = tot;
            tot += c;
        }
        s_base = tot ? atomicAdd(p.wl_hdr + wl_parity(p), tot) : 0;
    }
    __syncthreads();
    return s_base + s_warp[warp] + __popc(bal & ((1u << lane) - 1u));
}

}  // namespace pcgrl
