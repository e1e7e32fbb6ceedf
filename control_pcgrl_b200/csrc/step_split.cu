// Split env-step path for the bit-board problems: three launches per step instead of the fused kernel's one,
// so that every lane of every search warp has a grid to work on.
//
//   k_split_act    thread-per-env: representation update (single-byte scatter into the int8 grid), counters, done,
//                  zero reward for unchanged envs; envs whose map changed are appended (CTA-aggregated atomic) to a
//                  GLOBAL work list as (env, cell).
//   k_split_stats  the stat searches over the work list.  Two variants:
//       static  (any bit-board machine): a warp takes 32 consecutive items, stages their grids as bit-boards in
//               shared memory cooperatively, then every lane runs one from-scratch search -- full warps whatever
//               the per-tile change count was (the fused kernel's tiles hold 128 +- 8 changed envs for its 128
//               threads: the overflow items ran as a second round at 1-3 lanes per warp).
//       incremental (binary): the one changed cell only touches the components next to it.  From the per-env
//               cache (passable board, one far tile per non-isolated component, a cell of the component that
//               attains path-length) the machine floods the affected region U, redoes calc_longest_path's two
//               sweeps inside U only, and sweeps the untouched components too (in the same final sweep) only when
//               the one that held the maximum was touched; otherwise it skips the final sweep when the first sweeps
//               prove that it cannot beat the old path-length: 29 instead of 93 board expansions per changed grid on
//               16x16 narrow rollouts (scripts/inc_work_counts.py), bit-identical results (helper.py:255-276 is a
//               per-component computation; components the edit does not touch keep their first tile, far tile
//               and eccentricity).  Work per item is uneven (0..135 expansions), so lanes claim items one by one
//               from their warp's slice of the list instead of running in batches.
//   k_split_out    thread-per-changed-env: fp64 loss(new) - loss(old), stats / reward / packed record; the list is
//                  handed from step to step through ping-pong counters (see the header layout below).
//   k_step_inc     all three in ONE launch for mid-size shards.  step_lanegroup.cu holds the small-shard kernel.
//
// Reference path replaced: the same as step_bitboard.cu (envs/pcgrl_env.py:267-342, envs/reps/*_rep.py,
// envs/probs/binary/binary_prob.py:152-158, envs/probs/zelda/zelda_ctrl_prob.py:90-168, envs/helper.py:200-276,
// control_wrappers.py:216-244, 318-345).
#include "pcgrl_device.cuh"
#include "step_common.cuh"
#include "bitboard_machines.cuh"
#include "worklist.cuh"

namespace pcgrl {

constexpr int SPLIT_MIN_CTAS = 10;
constexpr int INC_CTAS_PER_SM = 6;       // 128-thread CTAs of the incremental search resident per SM (A/B 4 / 6 / 8 / 12 at
                                         // R=3: 0.412 / 0.393 / 0.384 / 0.378 ms per step; with the joint final sweep, 6 / 8 / 9:
                                         // 0.2686 / 0.2697 / 0.2712, profiles/r03_inc_joint_sweep.txt; with the skipped final
                                         // sweep, 6 / 8: 0.2576 / 0.2590 with claims of 12 lanes, 0.2549 / 0.2566 with claims of 8,
                                         // profiles/r04_inc_skip_final_sweep.txt)
constexpr int INC_CTAS_PER_SM_LOOKAHEAD = 8;   // the same for the search of the incremental lookahead, which keeps 8:
                                               // scripts/bench_lookahead.py, 8 / 6 CTAs per SM, binary-narrow lookahead_all
                                               // of 1 Mi envs 0.482-0.486 / 0.489 ms, binary-wide 512 actions of 16 Ki envs
                                               // 1.794-1.795 / 1.830-1.836 ms (profiles/r04_inc_skip_final_sweep.txt)
constexpr int INC_CTAS_PER_SM_HOST = 4;  // the same inside the host pipeline: most of the SM's registers stay free, so the
                                         // update / output kernels of the neighbouring chunks run next to the search
                                         // (e2e at 4 chunks, 2 / 3 / 4 / 5 / 8 CTAs per SM: 2.48 / 2.60 / 2.51 / 2.36 / 2.11e9 with the
                                         // copies on the compute streams; with separate copy streams 3 / 4 / 5 / 8:
                                         // 2.56 / 2.75 / 2.71 / 2.42e9, profiles/r02_e2e_cps_chunks_split.txt)
constexpr int INC_MIN_CLAIM = 8;         // lanes that must be waiting before a warp hands out new items: the claim / init
                                         // stream then runs with that many lanes (A/B 1 / 4 / 8 at R=3: 0.412 / 0.390 / 0.387; at
                                         // R=12, 8 / 12 / 16 / 24: 0.2978 / 0.2996 / 0.3022 / 0.3263 ms, profiles/r02_ab_inc_claim_window.txt;
                                         // with the joint final sweep 8 / 12: 0.2675 / 0.2697 in the split path,
                                         // profiles/r03_inc_joint_sweep.txt; with the skipped final sweep 8 / 12: 0.2566 / 0.2590 at 8
                                         // CTAs per SM, and k_step_inc (64 Ki envs, binary-wide + controls) 0.0596 / 0.0596 ms,
                                         // profiles/r04_inc_skip_final_sweep.txt)
constexpr int INC_EXPAND_R = 12;         // board expansions per trip.  Every trip also issues each transition stream that
                                         // some lane needs (flood done / next component / final sweep / finish, several
                                         // hundred instructions at 2-3 lanes), so few long trips beat many short ones although
                                         // lanes idle inside the window: A/B 2 / 3 / 4 / 6 / 8 / 12 -> 0.466 / 0.412 / 0.356 /
                                         // 0.325 / 0.308 / 0.303 ms per step (1 Mi envs, 8 CTAs per SM); 16 / 20 -> 0.3018 / 0.3140
                                         // against 0.2996 for 12 in a later run; with the joint final sweep 8 / 12 / 16 -> 0.2729 /
                                         // 0.2697 / 0.2733 (profiles/r03_inc_joint_sweep.txt); with the final sweep skipped under
                                         // the min(2 e1, |C| - 1) bound, 8 / 12 / 16 -> 0.2653 / 0.2599 / 0.2629
                                         // (profiles/r04_inc_skip_final_sweep.txt)
constexpr int EXPAND_R_SPLIT = 3;        // board expansions per trip of the static search (as in the fused kernel)

constexpr int ACT_THREADS = 256;
constexpr int STAT_THREADS = 128;
// threads per CTA of the static search: as many warps as keep the staged bit-boards under 48 KB of shared memory
__host__ __device__ constexpr int stat_threads(int bbw) { return bbw <= 96 ? 128 : 64; }
constexpr int OUT_THREADS = 256;
// ------------------------------------------------------------------------------------------------
// k_split_act
// IDX (pcgrl_step_envs): p.n_envs is the list length; thread j applies action row j to env env_idx[j] of the shard's
// n_src envs.  An index outside the shard loads and writes nothing and sets status bit 256.
// ------------------------------------------------------------------------------------------------
template <bool IDX>
__global__ void __launch_bounds__(ACT_THREADS) k_split_act(const KParams p, const int32_t* env_idx, int64_t n_src) {
    const int64_t j = (int64_t)blockIdx.x * ACT_THREADS + threadIdx.x;
    int64_t gid = j;
    bool need = false;
    int cell = -1;
    if (j < p.n_envs) {
        if constexpr (IDX) {
            gid = env_idx[j];
            if ((uint64_t)gid < (uint64_t)n_src) need = step_counters(p, gid, apply_action(p, j, gid, &cell));
            else if (p.status) atomicOr(p.status, 256);
        } else {
            need = step_counters(p, gid, apply_action(p, gid, &cell));
        }
    }
    const int slot = wl_append_slot<ACT_THREADS>(p, need);
    if (need) wl_items(p)[slot] = make_int2((int)gid, cell);
}

// ------------------------------------------------------------------------------------------------
// k_split_stats, static variant: one from-scratch search per lane, 32 consecutive list items per warp
// ------------------------------------------------------------------------------------------------
template <class Machine, int NW, bool TWO>
__global__ void __launch_bounds__(stat_threads(Machine::Prob::P * NW), NW <= 8 ? SPLIT_MIN_CTAS : 1)
k_split_stats(const KParams p) {
    using Prob = typename Machine::Prob;
    constexpr int P = Prob::P;
    constexpr int K = Prob::K;
    constexpr int BBW = P * NW;
    constexpr int THREADS = stat_threads(BBW);
    __shared__ uint32_t s_bb[THREADS * BBW];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int count = wl_count_search(p);
    const int first = (blockIdx.x * (THREADS / 32) + warp) * 32;
    if (first >= count) return;   // warps are independent: no CTA-wide barrier anywhere in this kernel
    const int n_here = min(32, count - first);
    const int2* items = wl_items(p) + first;
    uint32_t* wbb = s_bb + warp * 32 * BBW;

    // stage the warp's grids as per-plane bit-boards (as phase B of the fused kernel)
    stage_boards<Prob, NW, TWO, 32>(p, lane, n_here, wbb,
                                    [&](int slot) { return p.grids + (int64_t)items[slot].x * p.row_stride; });
    const bool mine = lane < n_here;
    const int64_t env = mine ? items[lane].x : 0;
    Machine m;
    if (mine) m.init(wbb + lane * BBW, p, env);
    int out[K];
    // One trip = EXPAND_R_SPLIT board expansions, then the transition stream for the lanes whose frontier
    // died.  The warp-wide vote at the top makes every lane start every trip together: without it the lanes that
    // loop back early run ahead of the ones in a transition, the warp falls apart into groups that never re-merge, and
    // both streams are issued once per group (ncu: transitions at 3.7 lanes, expansions at 19; 0.432 against 0.381 ms
    // per step).  Fixed windows: adaptive rounds (expand while a share of the running lanes is alive) measured
    // 0.42-0.59 ms against 0.38 -- waiting lanes cost more than the fuller transition stream saves.
    bool running = mine;
    for (;;) {
        if (!__any_sync(0xffffffffu, running)) break;
        bool dead = false;
        if (running) {
            bool alive = m.expand();
#pragma unroll
            for (int r = 1; r < EXPAND_R_SPLIT; ++r)
                if (alive) alive = m.expand();
            dead = !alive;
        }
        __syncwarp();
        if (dead && m.transition(out)) running = false;
    }
    if (!mine) return;
    int32_t* o = wl_stats(p) + (int64_t)(first + lane) * K;
#pragma unroll
    for (int k = 0; k < K; ++k) o[k] = out[k];
    if constexpr (Machine::HAS_CACHE)
        if (p.cache) m.store_cache((uint32_t*)(p.cache + env * p.cache_stride));
}

// ------------------------------------------------------------------------------------------------
// BinaryIncMachine: regions / path-length of a binary map after a one-cell edit, from the per-env cache.
//
// calc_num_regions (helper.py:200-210) counts components; calc_longest_path (:255-276) takes, per component in
// row-major order of its first tile, BFS(first tile) -> far tile (np.argmax: row-major-first maximum) -> BFS(far)
// and keeps the largest second-sweep maximum.  Both are sums / maxima of per-component terms, and a component the
// edit does not touch keeps its first tile, far tile and eccentricity.  With c the edited cell, D+ / D- the cells
// that became passable / solid (c or nothing), P' the new passable board:
//   U  = flood fill in P' from D+ and from the passable neighbours of D-   (every new component that is affected)
//   A  = U | D-                                          (covers every OLD component that is affected, entirely)
//   regions' = regions - #old components in A + #components of U
//              (#old in A = far tiles in A + old isolated cells in A: each non-isolated component owns one far tile)
//   path'    = max(two-sweep maximum inside U, maximum over the untouched components), where the latter is the
//              old path-length if the cached cell of a maximal component lies outside A.  Otherwise ONE sweep from
//              the far tiles of U and of the untouched components together gives both maxima at once: they are
//              different components, so a multi-source BFS takes max(lu, lold) levels instead of lu + lold.
//              In the first case the final sweep is skipped when the first sweeps already prove lu <= path: the
//              first sweep of component C_j of U reaches depth e1_j = ecc(first tile), so its far tile has
//              ecc <= 2 * e1_j; if max_j 2 * e1_j <= path, path and m stay.  (The tighter min(2 * e1_j, |C_j| - 1)
//              skips the sweep on 4 % more changed grids, but the popcounts it needs cost more than that: 0.2599
//              against 0.2591 ms per step, profiles/r04_inc_skip_final_sweep.txt.)
// Isolated cells are counted next to c only: with Q = P' \ {c} and iso(Q) its cells without a neighbour in Q,
//   c became solid:     old isolated in A = {c} if c has no neighbour in Q,  new isolated in U = N(c) & iso(Q)
//   c became passable:  old isolated in A = N(c) & iso(Q),  new isolated in U = {c} if c has no neighbour in Q
// (U is connected from c or from c's neighbours, so a cell of U without a neighbour in P_old or in P' can only have
// touched the rest of U through c).
// A Python restatement of this update is pinned by the CPU tests, edit by edit, on the from-scratch computation and on
// the two sweeps it replaced (same cache rows bit for bit, so the step paths can still share them), and
// tests/test_gpu_split.py checks every step of every env against pcgrl_stats recomputed from scratch.
// ------------------------------------------------------------------------------------------------
template <int NW, bool TWO>
struct BinaryIncMachine {
    static_assert(TWO, "the isolated-cell test reads 16-bit rows");
    using B = Board<NW, TWO>;
    static constexpr int SMEM_WORDS = 3 * NW;   // per thread: P' | U (non-isolated part) | far tiles of the rest
    uint32_t avail[NW], front[NW], fars[NW];
    uint32_t* sm;
    const uint32_t* cache;   // this env's cache row (still the OLD state until finish())
    int phase, level, regions, path, mcell, cell;   // path / mcell: the cache's path-length and m, old until the end
    bool hit;
    bool longer;    // phase 1: some far tile of U may have an eccentricity above path (else the final sweep is skipped)

    static __device__ __forceinline__ int lowest_pos(const uint32_t (&x)[NW]) {
        int pos = -1;   // branch-free: this runs in the few-lane transition stream
#pragma unroll
        for (int i = NW - 1; i >= 0; --i) {
            const int f = __ffs(x[i]);
            pos = f ? i * 32 + f - 1 : pos;
        }
        return pos;
    }

    // bitpos: bit position of the edited cell in the board (word * 32 + bit)
    __device__ __forceinline__ void init(uint32_t* smem, const uint32_t* c, int bitpos, int regions_old, int path_old) {
        sm = smem;
        cache = c;
        regions = regions_old;
        path = path_old;
        cell = bitpos;
        const uint4* c4 = (const uint4*)c;
        uint32_t pn[NW], d[NW], seed[NW];
        static_assert(NW % 4 == 0 || NW < 4, "cache rows are read as 128-bit vectors");
        if constexpr (NW >= 4) {
#pragma unroll
            for (int i = 0; i < NW / 4; ++i) {
                const uint4 v = c4[i];
                pn[4 * i] = v.x, pn[4 * i + 1] = v.y, pn[4 * i + 2] = v.z, pn[4 * i + 3] = v.w;
            }
        } else {
#pragma unroll
            for (int i = 0; i < NW; ++i) pn[i] = c[i];
        }
        mcell = (int)c[2 * NW];
        const int w = bitpos >> 5;
        const uint32_t bit = 1u << (bitpos & 31);
        uint32_t now_pass = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            d[i] = i == w ? bit : 0u;
            pn[i] ^= d[i];
            now_pass |= pn[i] & d[i];
            sm[i] = pn[i];
        }
        // seed of the flood: the cell itself if it became passable, else its passable neighbours
        B::expand_and(d, pn, seed);
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            front[i] = now_pass ? d[i] : seed[i];
            avail[i] = pn[i] & ~front[i];
            fars[i] = 0;
        }
        phase = 0;
        level = 0;
        hit = false;
        longer = false;
    }
    __device__ __forceinline__ bool expand() {
        uint32_t n[NW];
        if (!B::expand_and(front, avail, n)) return false;
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            avail[i] = B::minus_subset(avail[i], n[i]);
            front[i] = n[i];
        }
        ++level;
        return true;
    }
    // init for the list item (env, cell) of a map W cells wide: the cell's bit, and the env's cache row and old stats
    __device__ __forceinline__ void start(uint32_t* smem, const KParams& p, int64_t env, int cell_idx, int W) {
        const int y = cell_idx / W, x = cell_idx - y * W;
        const int32_t* st = p.stats + env * 2;
        init(smem, (const uint32_t*)(p.cache + env * p.cache_stride), B::bitpos(y, x), st[0], st[1]);
    }
    // the frontier died; returns true when the search is over (call finish())
    __device__ __forceinline__ bool transition() {
        if (phase == 0) {
            // flood done: U = P' \\ avail.  Account for the old components it swallowed, set up the sweeps inside U.
            int k_old = 0;
#pragma unroll
            for (int i = 0; i < NW; ++i) {
                const uint32_t fo = cache[NW + i];
                const uint32_t u = sm[i] & ~avail[i];
                const uint32_t rest = fo & avail[i];               // avail = P' \ U: far tiles of the untouched components
                k_old += __popc(fo ^ rest);                        // far tiles in A (fo lies in P_old, P_old \ A = P' \ U)
                sm[NW + i] = u;
                sm[2 * NW + i] = rest;
                avail[i] = u;
                front[i] = 0;
            }
            hit = mcell >= 0 && (mcell == cell || (sm[NW + (mcell >> 5)] >> (mcell & 31)) & 1u);   // m in U | D-
            // isolated cells next to c.  Rows y-2 .. y+2 of Q = P' \ {c} (c = (y, x) at word w, bit b; a word holds
            // rows 2w and 2w+1, so row y sits at bit 16 * (y & 1) = b & 16 of word w).
            const int w = cell >> 5, b = cell & 31, s = b & 16;
            const uint32_t bit = 1u << b, mx = 1u << (b & 15);
            const uint32_t pw = sm[w], q = pw & ~bit;
            const bool grew = pw & bit;
            const uint32_t qlo = w > 0 ? sm[w - 1] : 0u, qhi = w + 1 < NW ? sm[w + 1] : 0u;
            const uint32_t r01 = __funnelshift_r(qlo, q, s);       // rows y-2 | y-1 << 16
            const uint32_t r23 = __funnelshift_r(q, qhi, s);       // rows y   | y+1 << 16
            const uint32_t r2 = r23 & 0xFFFFu;
            const uint32_t x13 = (r01 >> 16) | (r23 & 0xFFFF0000u);   // rows y-1 | y+1 << 16
            const uint32_t v13 = (r01 & 0xFFFFu) | r2 * 0x10001u | ((qhi >> s) << 16);   // their vertical neighbours
            const uint32_t iso13 = x13 & ~(v13 | ((x13 + x13) & 0xFFFEFFFEu) | ((x13 >> 1) & 0x7FFF7FFFu));
            const uint32_t iso2 = r2 & ~((x13 | x13 >> 16) | (r2 << 1) | (r2 >> 1));
            const uint32_t nb13 = mx * 0x10001u, nb2 = (mx << 1) | (mx >> 1);   // c's neighbours in those rows
            const uint32_t up = iso13 & nb13 & 0xFFFFu, dn = (iso13 & nb13) >> 16, lr = iso2 & nb2;
            const int n_iso = (up != 0) + (dn != 0) + __popc(lr);
            const bool alone = !((x13 & nb13) | (r2 & nb2));
            // the new isolated cells of U leave it: c, or the isolated neighbours of c (rows y-1 | y | y+1 back at
            // their words w-1, w, w+1)
            uint32_t cl_lo = 0, cl_mid, cl_hi = 0;
            if (grew) {
                cl_mid = alone ? bit : 0u;
                regions += alone - n_iso;
            } else {
                const uint32_t rows = up | (lr << 16);
                cl_lo = s ? 0u : rows << 16;
                cl_mid = s ? rows : __funnelshift_l(rows, dn, 16);
                cl_hi = s ? dn : 0u;
                regions += n_iso - alone;
            }
            regions -= k_old;
            if (cl_lo | cl_mid | cl_hi) {
                if (cl_lo) sm[NW + w - 1] &= ~cl_lo;
                sm[NW + w] &= ~cl_mid;
                if (cl_hi) sm[NW + w + 1] &= ~cl_hi;
#pragma unroll
                for (int i = 0; i < NW; ++i) avail[i] = sm[NW + i];
            }
            phase = 1;
            level = 0;
        }
        if (phase == 1) {   // first sweeps inside U, one component at a time (BinaryMachine phase 0)
            // the component whose sweep just died (none on entry from phase 0: level 0) reached depth e1 = level
            longer |= 2 * level > path;
            uint32_t t[NW];
            B::minus_one(front, t);
#pragma unroll
            for (int i = 0; i < NW; ++i) fars[i] |= front[i] & ~t[i];
            if (B::minus_one(avail, t)) {
#pragma unroll
                for (int i = 0; i < NW; ++i) {
                    front[i] = avail[i] & ~t[i];
                    avail[i] &= t[i];
                }
                ++regions;
                level = 0;
                return false;
            }
            // final sweep: from the far tiles of U, and when the component that held the maximum was touched, from
            // those of the untouched components too (isolated cells may stay in avail: the sweep never reaches them).
            // Untouched: path' = max(path, lu), and the first sweeps bound lu by path -- nothing to sweep.
            phase = 2;
            if (!hit && !longer) return true;
            uint32_t any = 0;
#pragma unroll
            for (int i = 0; i < NW; ++i) {
                front[i] = fars[i] | (hit ? sm[2 * NW + i] : 0u);
                avail[i] = sm[i] & ~front[i];
                any |= front[i];
            }
            level = 0;
            if (any) return false;
        }
        // the final sweep died (or had no sources)
        if (hit) {      // the maximum over all components; on a tie the untouched ones keep m, as before the edit
            uint32_t rest[NW];
#pragma unroll
            for (int i = 0; i < NW; ++i) rest[i] = front[i] & ~sm[NW + i];
            const int mr = lowest_pos(rest);
            mcell = mr >= 0 ? mr : lowest_pos(front);
            path = level;
        } else if (level > path) {
            mcell = lowest_pos(front);
            path = level;
        }
        return true;
    }
    // results + the new cache row
    __device__ __forceinline__ void finish(int* out, uint32_t* c) const {
        results(out);
        store_cache(c);
    }
    __device__ __forceinline__ void results(int* out) const {
        out[0] = regions;
        out[1] = path;
    }
    __device__ __forceinline__ void store_cache(uint32_t* c) const {
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            c[i] = sm[i];
            c[NW + i] = sm[2 * NW + i] | fars[i];
        }
        c[2 * NW] = (uint32_t)mcell;
    }
};

// ------------------------------------------------------------------------------------------------
// k_split_stats, incremental variant: persistent-size grid, every warp owns a contiguous slice of the work list
// and its lanes claim items from it one by one (ballot-ranked at a convergent point, no atomics).  Static slices:
// fetching items from a global counter instead did not move the bench line (0.2909 against 0.2913 ms per step) and
// cut e2e from 2.60 to 2.51e9 (profiles/r02_ab_inc_dynamic.txt).  Fixed windows of INC_EXPAND_R expansions:
// adaptive rounds measured 0.334 ms against 0.303.
// LOOKAHEAD (lookahead.cu): the items are candidate edits of unchanged envs; the cache rows are read, never written.
// ------------------------------------------------------------------------------------------------
template <int NW, bool TWO, bool LOOKAHEAD = false>
__global__ void __launch_bounds__(STAT_THREADS) k_split_stats_inc(const KParams p) {
    using M = BinaryIncMachine<NW, TWO>;
    __shared__ uint32_t s_work[STAT_THREADS * M::SMEM_WORDS];
    const int tid = threadIdx.x, lane = tid & 31;
    const int count = wl_count_search(p);
    const int n_warps = gridDim.x * (STAT_THREADS / 32);
    const int gw = blockIdx.x * (STAT_THREADS / 32) + (tid >> 5);
    const int per = (count + n_warps - 1) / n_warps;
    int lo = min(count, gw * per);
    const int hi = min(count, lo + per);
    if (lo >= hi) return;
    const int2* items = wl_items(p);
    int32_t* stats_out = wl_stats(p);
    const int W = p.d1;
    M m;
    bool active = false;
    int item = 0;
    int64_t env = 0;
    for (;;) {
        const unsigned need = __ballot_sync(0xffffffffu, !active);
        if (need && lo < hi && (__popc(need) >= INC_MIN_CLAIM || need == 0xffffffffu || hi - lo < INC_MIN_CLAIM)) {
            const int mine = lo + __popc(need & ((1u << lane) - 1u));
            if (!active && mine < hi) {
                item = mine;
                const int2 it = items[item];
                env = it.x;
                m.start(s_work + tid * M::SMEM_WORDS, p, env, it.y, W);
                active = true;
            }
            lo = min(hi, lo + __popc(need));
        }
        const unsigned act = __ballot_sync(0xffffffffu, active);
        if (!act) break;
        if (active) {
            bool alive = m.expand();
#pragma unroll
            for (int r = 1; r < INC_EXPAND_R; ++r)
                if (alive) alive = m.expand();
            if (!alive && m.transition()) {
                int out[2];
                if constexpr (LOOKAHEAD) m.results(out);
                else m.finish(out, (uint32_t*)(p.cache + env * p.cache_stride));
                *(int2*)(stats_out + (int64_t)item * 2) = make_int2(out[0], out[1]);
                active = false;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_step_inc: the whole binary env step in ONE launch around the incremental search (no global work list).
// Every warp owns a contiguous slice of the shard's envs and loops over three kinds of work, each issued with
// (nearly) all 32 lanes:
//   update  the next 32 envs of the slice: representation update, counters, done, zero reward for unchanged
//           maps (thread-per-env, as k_split_act); the changed ones go into the warp's item ring in shared memory;
//   search  lanes pick items from the ring as they become free (at least INC_MIN_CLAIM at a time) and run
//           BinaryIncMachine trips; a finished lane writes its env's cache row and parks (env, regions,
//           path-length) in the warp's result ring;
//   output  once 32 results wait (or nothing else is left): one lane per result does the fp64 reward and writes
//           stats / reward / packed record (as k_split_out).
// The update and output passes are memory-latency work; in the split path they were two separate kernels (42 +
// 30 us of the 303 us step at 1 Mi envs) during which the ALU pipes idled, here other warps' searches cover them.
// ------------------------------------------------------------------------------------------------
constexpr int STEP_INC_MIN_CTAS = 6;
constexpr int STEP_INC_ROUNDS = 1;   // update rounds (of 32 envs) per warp the grid is sized for below 48 Ki envs, see launch_split
template <int NW, bool TWO>
__global__ void __launch_bounds__(STAT_THREADS, STEP_INC_MIN_CTAS) k_step_inc(const __grid_constant__ KParams p) {
    using M = BinaryIncMachine<NW, TWO>;
    constexpr int WARPS = STAT_THREADS / 32;
    constexpr int RING = 64;
    __shared__ uint32_t s_work[STAT_THREADS * M::SMEM_WORDS];
    __shared__ int2 s_items[WARPS][RING];     // (env, cell) waiting for a lane
    __shared__ int4 s_res[WARPS][RING];       // (env, regions, path-length, -) waiting for the output pass
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const int64_t n_warps = (int64_t)gridDim.x * WARPS;
    const int64_t gw = (int64_t)blockIdx.x * WARPS + warp;
    const int64_t per = ((p.n_envs + n_warps - 1) / n_warps + 31) / 32 * 32;
    int64_t e_next = min(p.n_envs, gw * per);
    const int64_t e_hi = min(p.n_envs, e_next + per);
    if (e_next >= e_hi) return;
    int2* items = s_items[warp];
    int4* res = s_res[warp];
    const int W = p.d1;
    int it_head = 0, it_cnt = 0, res_head = 0, res_cnt = 0;     // warp-uniform
    M m;
    bool active = false;
    int64_t env = 0;
    for (;;) {
        // ---- update: refill the item ring from the warp's env slice
        if (it_cnt < 32 && e_next < e_hi) {
            const int64_t gid = e_next + lane;
            int cell = -1;
            const bool need = gid < e_hi && inc_update_env(p, gid, &cell);
            const unsigned bal = __ballot_sync(0xffffffffu, need);
            if (need) items[(it_head + it_cnt + __popc(bal & lt)) & (RING - 1)] = make_int2((int)gid, cell);
            it_cnt += __popc(bal);
            e_next += 32;
            __syncwarp();
        }
        const bool drained = e_next >= e_hi;
        // ---- hand items to free lanes
        const unsigned idle = __ballot_sync(0xffffffffu, !active);
        if (idle && it_cnt > 0 && (__popc(idle) >= INC_MIN_CLAIM || idle == 0xffffffffu || drained)) {
            const int rank = __popc(idle & lt);
            if (!active && rank < it_cnt) {
                const int2 it = items[(it_head + rank) & (RING - 1)];
                env = it.x;
                m.start(s_work + tid * M::SMEM_WORDS, p, env, it.y, W);
                active = true;
            }
            const int taken = min(__popc(idle), it_cnt);
            it_head += taken;
            it_cnt -= taken;
        }
        const unsigned act = __ballot_sync(0xffffffffu, active);
        // ---- output: 32 results at a time, or whatever is left at the end
        if (res_cnt >= 32 || (res_cnt > 0 && !act && it_cnt == 0 && drained)) {
            const int n_out = min(32, res_cnt);
            if (lane < n_out) {
                const int4 r = res[(res_head + lane) & (RING - 1)];
                inc_output_env(p, r.x, r.y, r.z);
            }
            res_head += n_out;
            res_cnt -= n_out;
            __syncwarp();
        }
        if (!act) {
            if (it_cnt == 0 && drained && res_cnt == 0) break;
            continue;
        }
        // ---- search: one trip of every active lane
        bool finished = false;
        int out[2] = {0, 0};
        if (active) {
            bool alive = m.expand();
#pragma unroll
            for (int r = 1; r < INC_EXPAND_R; ++r)
                if (alive) alive = m.expand();
            if (!alive && m.transition()) {
                m.finish(out, (uint32_t*)(p.cache + env * p.cache_stride));
                finished = true;
                active = false;
            }
        }
        const unsigned fin = __ballot_sync(0xffffffffu, finished);
        if (finished) res[(res_head + res_cnt + __popc(fin & lt)) & (RING - 1)] = make_int4((int)env, out[0], out[1], 0);
        res_cnt += __popc(fin);
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// k_split_out
// ------------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(OUT_THREADS) k_split_out(const KParams p) {
    const int count = *(volatile const int*)(p.wl_hdr + 4);
    const int i = blockIdx.x * OUT_THREADS + threadIdx.x;
    if (i == 0) p.wl_hdr[3] = p.wl_hdr[3] + 1;   // the next step uses the other counter (no CTA of this kernel reads [3])
    if (i < count) {
        const int64_t env = wl_items(p)[i].x;
        int32_t nw[K];
        const int32_t* o = wl_stats(p) + (int64_t)i * K;
#pragma unroll
        for (int k = 0; k < K; ++k) nw[k] = o[k];
        finish_env<K>(p, env, nw);
    }
}

// ------------------------------------------------------------------------------------------------
// host-side dispatch
// ------------------------------------------------------------------------------------------------
// resident CTAs per SM of the persistent incremental kernels
static int inc_ctas_per_sm(bool host_chunk) { return host_chunk ? INC_CTAS_PER_SM_HOST : INC_CTAS_PER_SM; }

// env_idx (pcgrl_step_envs): the list of p.n_envs env indices into a shard of n_src envs (path SPLIT or INC).
template <class Machine, int NW, bool TWO>
static cudaError_t launch_split(const KParams& p, cudaStream_t s, StepPath path, const int32_t* env_idx,
                                int64_t n_src) {
    constexpr int K = Machine::Prob::K;
    const int64_t n = p.n_envs;
    if (n == 0) return cudaSuccess;
    cudaError_t e;
    if constexpr (Machine::HAS_CACHE && TWO) {
        if (path == INC_FUSED) {     // the whole step in one launch (k_step_inc)
            int n_sm = 0;
            if ((e = sm_count(n_sm)) != cudaSuccess) return e;
            // envs per warp = 32 * m.  A warp's first 32 envs yield ~16 changed ones, i.e. half-empty warps for the whole
            // search; with two update rounds per warp the ring refills and every lane gets an item.  And the grid is
            // sized so that EVERY CTA gets work: with the plain cap (6 CTAs per SM) a 128 Ki-env shard ran 64 envs per warp
            // on 512 of its 888 CTAs while the others exited at once.  A/B of m (profiles/r02_step_inc_rounds.txt, kernel
            // ms, m = 1 / 2 / 3 / 4): 32 Ki envs 0.042 / 0.048 / 0.062 / 0.075, 64 Ki 0.060 / 0.056 / 0.070 / 0.077,
            // 128 Ki 0.095 / 0.075 / 0.083 / 0.089.
            const int64_t cap = (int64_t)n_sm * inc_ctas_per_sm(p.host_chunk != 0);
            int64_t m = n >= (48 << 10) ? 2 : STEP_INC_ROUNDS;
            const int64_t need_m = (n + STAT_THREADS * cap - 1) / (STAT_THREADS * cap);
            if (m < need_m) m = need_m;
            const int64_t want = (n + STAT_THREADS * m - 1) / (STAT_THREADS * m);
            k_step_inc<NW, TWO><<<(unsigned)(want < cap ? want : cap), STAT_THREADS, 0, s>>>(p);
            return cudaGetLastError();
        }
    }
    const unsigned act_blocks = (unsigned)((n + ACT_THREADS - 1) / ACT_THREADS);
    if (env_idx) k_split_act<true><<<act_blocks, ACT_THREADS, 0, s>>>(p, env_idx, n_src);
    else k_split_act<false><<<act_blocks, ACT_THREADS, 0, s>>>(p, nullptr, 0);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    bool ran_inc = false;
    if constexpr (Machine::HAS_CACHE && TWO) {
        if (path == INC) {
            int n_sm = 0;
            if ((e = sm_count(n_sm)) != cudaSuccess) return e;
            const int64_t want = (n + STAT_THREADS - 1) / STAT_THREADS;
            const int64_t cap = (int64_t)n_sm * inc_ctas_per_sm(p.host_chunk != 0);
            k_split_stats_inc<NW, TWO><<<(unsigned)(want < cap ? want : cap), STAT_THREADS, 0, s>>>(p);
            ran_inc = true;
        }
    }
    if (!ran_inc) {
        constexpr int T = stat_threads(Machine::Prob::P * NW);
        k_split_stats<Machine, NW, TWO><<<(unsigned)((n + T - 1) / T), T, 0, s>>>(p);
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    k_split_out<K><<<(unsigned)((n + OUT_THREADS - 1) / OUT_THREADS), OUT_THREADS, 0, s>>>(p);
    return cudaGetLastError();
}

template <template <int, bool> class Machine>
static cudaError_t dispatch_split(const KParams& p, cudaStream_t s, StepPath path, bool& supported,
                                  const int32_t* env_idx, int64_t n_src) {
    supported = false;
    if (p.ndim != 2) return cudaSuccess;
    return with_board(p.d0, p.d1, supported, [&](auto b) {
        using B = decltype(b);
        return launch_split<Machine<B::WORDS, B::TWO_ROWS>, B::WORDS, B::TWO_ROWS>(p, s, path, env_idx, n_src);
    });
}

// MODE_STEP of a bit-board problem through the split path: `path` is SPLIT, INC or INC_FUSED, and a shard without a
// search cache runs SPLIT (StepPath).  *n_launches = kernels launched.
// env_idx (pcgrl_step_envs, SPLIT / INC): step only the p.n_envs listed envs of a shard of n_src envs, through the
// shard's own work list; the search and output kernels address envs through the list items as for a full step.
cudaError_t launch_bitboard_split(const KParams& p, int problem, cudaStream_t s, StepPath path, bool& supported,
                                  int& n_launches, const int32_t* env_idx, int64_t n_src) {
    supported = false;
    n_launches = 3;
    if (p.mode != MODE_STEP || !p.worklist || p.rep == PCGRL_REP_CELLULAR) return cudaSuccess;
    if (problem == PCGRL_PROB_BINARY) {
        if (!p.cache || p.d0 > 16 || p.d1 > 16) path = SPLIT;
        if (path == INC_FUSED) n_launches = 1;
        return dispatch_split<BinaryMachine>(p, s, path, supported, env_idx, n_src);
    }
    if (problem == PCGRL_PROB_ZELDA) return dispatch_split<ZeldaMachine>(p, s, SPLIT, supported, env_idx, n_src);
    if (problem == PCGRL_PROB_BINARY_HOLEY) {
        supported = p.ndim == 2 && p.d1 + 2 <= 32 && p.d0 + 2 <= 32;
        if (!supported) return cudaSuccess;
        if (p.d0 + 2 <= 18) return launch_split<BinaryHoleyMachine<18, false>, 18, false>(p, s, SPLIT, env_idx, n_src);
        return launch_split<BinaryHoleyMachine<32, false>, 32, false>(p, s, SPLIT, env_idx, n_src);
    }
    return cudaSuccess;
}

// The search kernel of the incremental lookahead (lookahead.cu): the work list of p holds (env, cell) candidate
// edits, p.stats / p.cache are the shard's.  Sized as the split path's search, with INC_CTAS_PER_SM_LOOKAHEAD.
cudaError_t launch_lookahead_search(const KParams& p, cudaStream_t s) {
    int n_sm = 0;
    cudaError_t e = sm_count(n_sm);
    if (e != cudaSuccess) return e;
    const int64_t want = (p.n_envs + STAT_THREADS - 1) / STAT_THREADS;
    const int64_t cap = (int64_t)n_sm * INC_CTAS_PER_SM_LOOKAHEAD;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    bool supported = false;
    e = with_board(p.d0, p.d1, supported, [&](auto b) {
        using B = decltype(b);
        if constexpr (!B::TWO_ROWS) {
            return cudaErrorInvalidValue;   // a shard with a search cache has maps of at most 16x16
        } else {
            k_split_stats_inc<B::WORDS, true, true><<<grid, STAT_THREADS, 0, s>>>(p);
            return cudaGetLastError();
        }
    });
    return supported ? e : cudaErrorInvalidValue;
}

// bytes per env of the incremental search cache (0: this config has none)
int bitboard_cache_stride(int problem, int ndim, int d0, int d1, int rep, int action_kind) {
    if (problem != PCGRL_PROB_BINARY || ndim != 2 || d0 > 16 || d1 > 16) return 0;
    if (rep == PCGRL_REP_CELLULAR || action_kind == PCGRL_ACT_PATCH) return 0;   // whole-map / multi-cell edits
    bool supported = false;
    return with_board(d0, d1, supported, [](auto b) { return (2 * decltype(b)::WORDS + 4) * 4; });
}

}  // namespace pcgrl
