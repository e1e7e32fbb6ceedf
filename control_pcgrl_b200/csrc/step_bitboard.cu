// Fused batched env-step kernel for the bit-board problems (maps up to 32x32):
//   representation update -> get_stats -> ControlWrapper reward, one launch for the whole env shard.
//
// Reference path replaced (paths relative to /root/reference/control_pcgrl/):
//   envs/pcgrl_env.py:267-342 (step), envs/reps/{narrow,turtle,wide,ca}_rep.py (update),
//   envs/probs/binary/binary_prob.py:152-158, envs/probs/zelda/zelda_ctrl_prob.py:90-168 (get_stats),
//   envs/helper.py:200-276 (calc_num_regions, run_dijkstra, calc_longest_path),
//   control_wrappers.py:216-244,318-345 (reward = loss - last_loss).
//
// Work decomposition per CTA (TILE consecutive envs):
//   A  thread-per-env: apply the action to the int8 grid in HBM (single-byte scatter, or whole-map rewrite
//      for the cellular rep), advance counters, decide done, flag envs whose map changed;
//   B  all threads: 128-bit coalesced loads of the changed grids, packed into per-plane bit-boards in
//      shared memory (one bit per cell; a "plane" is a set of tile codes);
//   C  thread-per-grid: every thread pulls changed envs from a shared-memory queue and runs the stat
//      searches as level-synchronous bit-board BFS held entirely in registers (NW 32-bit words): shifts
//      inside a word for x+-1, funnel shifts between neighbouring words for y+-1, no cross-lane traffic;
//   D  thread-per-env: fp64 loss(new stats) - loss(old stats), write stats / reward / done / counters.
#include "pcgrl_device.cuh"
#include "step_common.cuh"
#include "bitboard_machines.cuh"

namespace pcgrl {

constexpr int THREADS = 128;
constexpr int MIN_CTAS = 10;   // boards of <= 8 words: 48 registers, 10 CTAs (40 warps) per SM; A/B 1 / 10 -> 2.88 / 2.95e9
constexpr int EXPAND_R = 3;
constexpr int TILE8 = 256;     // envs per CTA when a board is <= 8 words (binary 16x16); A/B: 2 envs per thread is best
// envs per CTA, bounded so the shared-memory bit-boards stay under the 48 KB static limit
__host__ __device__ constexpr int tile_for(int bbw) { return bbw == 8 ? TILE8 : bbw < 8 ? 256 : (bbw <= 32 ? 256 : (bbw <= 80 ? 128 : 64)); }

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
template <class Machine, int NW, bool TWO>
__global__ void __launch_bounds__(THREADS, NW <= 8 ? MIN_CTAS : 1) k_step_bitboard(const KParams p) {
    using Prob = typename Machine::Prob;
    constexpr int P = Prob::P;
    constexpr int K = Prob::K;
    constexpr int BBW = P * NW;  // board words per env
    constexpr int TILE = tile_for(BBW);
    static_assert(TILE % 32 == 0 && THREADS % 32 == 0, "phase_a's warp ballots need every lane of a warp in the same trip");

    __shared__ uint32_t s_bb[TILE * BBW];
    __shared__ int32_t s_stats[TILE * K];
    __shared__ int16_t s_list[TILE];   // compact list of tile-local env indices that need stats
    __shared__ int16_t s_slot[TILE];   // env -> position in s_list, or -1
    __shared__ uint8_t s_flag[TILE];   // cellular: map changed
    __shared__ int s_count, s_next;

    // One CTA per tile.  (A persistent grid with a device-side tile counter, as in step_search.cuh, was A/B-tested
    // here and ran 2 % slower: the extra barriers cost more than the partly filled last wave.)
    const int tid = threadIdx.x;
    const int64_t base = (int64_t)blockIdx.x * TILE;
    const int64_t n_total = p.n_envs;
    const int tile_n = (int)min((int64_t)TILE, n_total - base);
    const int8_t* grids_in = (p.mode == MODE_STATS) ? p.stats_grids : p.grids;

    if (tid == 0) {
        s_count = 0;
        s_next = 0;
    }
    for (int e = tid; e < TILE; e += THREADS) {
        s_slot[e] = -1;
        s_flag[e] = 0;
    }
    __syncthreads();

    // ---------------- phase A: representation update / reset, counters, change flag ----------------
    phase_a<THREADS, TILE>(p, base, tile_n, s_list, s_slot, s_flag, &s_count);
    const int M = s_count;

    // ---------------- phase B: coalesced 128-bit grid loads -> per-plane bit-boards in smem --------
    // 16 cells (one uint4) are turned into a 16-bit membership mask per plane with SIMD-in-register ops:
    // a PRMT table lookup maps 4 tile codes to 4 0/1 bytes, a multiply gathers them into a nibble.
    stage_boards<Prob, NW, TWO, THREADS>(p, tid, M, s_bb,
                                         [&](int slot) { return grids_in + (base + s_list[slot]) * p.row_stride; });

    // ---------------- phase C: thread-per-grid stat searches, dynamic queue --------------------------
    // Each thread pulls the next changed env from the shared-memory queue as soon as it finishes one, so
    // lanes with short searches do not idle behind long ones; the search itself is a flat loop (one board
    // expansion per trip) so lanes in different phases of different grids execute the same instructions.
    // Fixed windows of EXPAND_R expansions: adaptive rounds (expand while a share of the warp's lanes is
    // alive) measured 0.45-0.60 ms per step against 0.385, and a warp-wide vote that starts every trip together
    // 0.393 against 0.385 (it pays in the split kernel, step_split.cu).
    {
        Machine m;
        int item = atomicAdd(&s_next, 1);
        bool active = item < M;
        if (active) m.init(s_bb + item * BBW, p, base + s_list[item]);
        while (active) {
            int out[K];
            // EXPAND_R expansions per trip: the transition stream (a few lanes) is then paid once per R
            // expansions of the warp instead of once per expansion; a lane whose frontier dies early idles for
            // the rest of the trip
            bool alive = m.expand();
#pragma unroll
            for (int r = 1; r < EXPAND_R; ++r)
                if (alive) alive = m.expand();
            if (alive) continue;
            if (m.transition(out)) {
#pragma unroll
                for (int k = 0; k < K; ++k) s_stats[item * K + k] = out[k];
                if constexpr (Machine::HAS_CACHE)
                    if (p.cache && p.mode != MODE_STATS)
                        m.store_cache((uint32_t*)(p.cache + (base + s_list[item]) * p.cache_stride));
                item = atomicAdd(&s_next, 1);
                active = item < M;
                if (active) m.init(s_bb + item * BBW, p, base + s_list[item]);
            }
        }
    }
    __syncthreads();

    // ---------------- phase D: reward (fp64), stats / outputs --------------------------------------
    phase_d<THREADS, K>(p, base, tile_n, s_slot, s_stats);
}

// ------------------------------------------------------------------------------------------------
// host-side dispatch
// ------------------------------------------------------------------------------------------------
template <class Machine, int NW, bool TWO>
static cudaError_t launch(const KParams& p, cudaStream_t s) {
    constexpr int TILE = tile_for(Machine::Prob::P * NW);
    const int64_t ctas = (p.n_envs + TILE - 1) / TILE;
    if (ctas == 0) return cudaSuccess;
    k_step_bitboard<Machine, NW, TWO><<<(unsigned)ctas, THREADS, 0, s>>>(p);
    return cudaGetLastError();
}

template <template <int, bool> class Machine>
static cudaError_t dispatch_shape(const KParams& p, cudaStream_t s, bool& supported) {
    supported = false;
    if (p.ndim != 2) return cudaSuccess;
    return with_board(p.d0, p.d1, supported, [&](auto b) {
        using B = decltype(b);
        return launch<Machine<B::WORDS, B::TWO_ROWS>, B::WORDS, B::TWO_ROWS>(p, s);
    });
}

cudaError_t launch_bitboard(const KParams& p, int problem, cudaStream_t s, bool& supported) {
    if (problem == PCGRL_PROB_BINARY) return dispatch_shape<BinaryMachine>(p, s, supported);
    if (problem == PCGRL_PROB_BINARY_HOLEY) {
        // the bordered board: H + 2 rows of W + 2 cells, one row per word
        supported = p.ndim == 2 && p.d1 + 2 <= 32 && p.d0 + 2 <= 32;
        if (!supported) return cudaSuccess;
        if (p.d0 + 2 <= 18) return launch<BinaryHoleyMachine<18, false>, 18, false>(p, s);
        return launch<BinaryHoleyMachine<32, false>, 32, false>(p, s);
    }
    if (problem == PCGRL_PROB_ZELDA) return dispatch_shape<ZeldaMachine>(p, s, supported);
    supported = false;
    return cudaSuccess;
}

}  // namespace pcgrl
