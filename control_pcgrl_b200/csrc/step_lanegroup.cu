// Lane-group env step for SMALL binary shards: NW lanes per level grid, one board word (two 16-cell rows) per lane.
//
// The thread-per-grid kernels (step_bitboard.cu, step_split.cu) keep a whole 16x16 board in one thread's registers:
// ~50 instructions per BFS level, ~35 levels and a handful of transitions per changed grid.  On a big shard that is
// what fills the integer pipes; a small shard (RLlib-scale batches) leaves the GPU far from full and its step lasts as
// long as the dependent chain of its WORST grid (~200 levels over the flood and the sweeps of a map with long
// corridors).  Here a grid's board is spread over NW lanes (NW = rows / 2: 8 lanes for 16x16), so a BFS level is ~14
// instructions per lane -- x+-1 inside the word, y+-1 inside the word as a 16-bit rotate, y+-1 across words as two
// width-NW shuffles -- and component bookkeeping (lowest cell, popcount sums, frontier tests) is a ballot / butterfly
// over the group.  Measured (profiles/r02_lanegroup_by_size.txt, profiles/r02_small_shard_ncu_summary.txt): a level
// costs a shuffle round trip (~55 cycles) instead of ~120-200 cycles of one thread's ALU chain; kernel time 24.9 / 27.1 /
// 31.5 us against 30.8 / 32.6 / 33.7 us for k_step_inc at 1 Ki / 4 Ki / 16 Ki envs, and a loss from 64 Ki envs on (4 grids
// per warp-instruction against 11-14), so pcgrl_step takes this kernel below 24 Ki envs only (api.cu, step_path()).
//
// One warp steps a tile of T consecutive envs (T = 8, 16 or 32, chosen so that the grid still fills the GPU):
//   update   thread-per-env representation update, counters, done (as k_split_act); ballot of the changed envs
//   search   the warp's 32 / NW lane groups take the changed envs one by one (ballot-ranked, no atomics) and run the
//            incremental search of step_split.cu's BinaryIncMachine -- the same algebra (flood U from the edit,
//            two sweeps inside U, re-sweep of the untouched components only if the maximal one was hit), restated
//            for one word per lane; the group's lanes write the env's new cache row
//   output   thread-per-env fp64 reward, stats, packed record (as k_split_out)
// in ONE launch, no global work list.  Reads and writes the same per-env cache as the other incremental paths, so
// a shard may switch between them from step to step (tests/test_gpu_split.py runs all of them side by side).
//
// Reference path replaced: the same as step_split.cu (envs/pcgrl_env.py:267-342, envs/reps/*_rep.py,
// envs/probs/binary/binary_prob.py:152-158, envs/helper.py:200-276, control_wrappers.py:216-244, 318-345).
#include "pcgrl_device.cuh"
#include "step_common.cuh"

namespace pcgrl {

constexpr int LG_EXPAND_R = 12;   // BFS levels per trip (computed blind, see expand_window).  A/B 4 / 6 / 8 / 12 (kernel time, CUDA
                                  // events): 2 Ki envs 28.8 / 26.4 / 25.7 / 25.0 us, 16 Ki envs 34.9 / 32.4 / 31.8 / 31.5 us -- a small
                                  // shard has issue slots to spare, so few long trips beat many short ones
constexpr int LG_THREADS = 128;

// Every collective below (shuffle, ballot) is issued by ALL 32 lanes with the full mask at warp-uniform points of the
// control flow, and the groups that have no use for the result simply do not commit it.  (The first version let every
// group run its own branch with a group-sized member mask: correct, but ptxas guards each sub-warp-mask collective with
// BRA.DIV and, whenever ANY lane of the warp sits in another branch, detours through WARPSYNC.COLLECTIVE -- 0.113 ms
// per step at 64 Ki envs against 0.065 for the thread-per-grid kernel.)
template <int NW>
struct LaneGroupInc {
    static constexpr unsigned FULL = 0xffffffffu;
    // per lane: one word of each board
    uint32_t pn, po, fo, avail, front, fars, unon, farrest;
    // group-uniform scalars (every lane of the group holds the same value)
    int phase, level, regions, lu, mcu, mold, lold;
    bool hit;
    unsigned gmask;     // the group's lanes within the warp
    int j;              // lane within the group = board word
    int lane;

    __device__ __forceinline__ bool gany(bool pred) const { return (__ballot_sync(FULL, pred) & gmask) != 0u; }
    __device__ __forceinline__ int gsum(int v) const {
#pragma unroll
        for (int o = NW / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
        return v;
    }
    // 4-neighbourhood of the cells of x (not masked by anything)
    __device__ __forceinline__ uint32_t nbr(uint32_t x) const {
        const uint32_t h = ((x << 1) & 0xFFFEFFFEu) | ((x >> 1) & 0x7FFF7FFFu);
        const uint32_t v = __funnelshift_l(x, x, 16);           // the two rows of the word swap: y+1 of the low row, y-1 of the high row
        uint32_t up = 0, dn = 0;
        if constexpr (NW > 1) {
            up = __shfl_up_sync(FULL, x, 1, NW) >> 16;           // high row of the word before -> above my low row
            dn = __shfl_down_sync(FULL, x, 1, NW) << 16;         // low row of the word after -> below my high row
            if (j == 0) up = 0;
            if (j == NW - 1) dn = 0;
        }
        return h | v | up | dn;
    }
    // bit position (word * 32 + bit) of the lowest cell of the group's board x, -1 if empty; *one = that cell as a
    // one-hot word on the lane that holds it (0 elsewhere)
    __device__ __forceinline__ int lowest(uint32_t x, uint32_t* one) const {
        const unsigned b = __ballot_sync(FULL, x != 0u) & gmask;
        const int first = __ffs(b) - 1;                          // warp lane index, -1 if none
        *one = lane == first ? (x & (0u - x)) : 0u;
        const int bit = __shfl_sync(FULL, __ffs(x) - 1, first < 0 ? lane : first);
        return first < 0 ? -1 : (first - (lane - j)) * 32 + bit;
    }

    // Start the search of an env for the groups with `go` (all lanes call; c / bitpos / stats only matter where go)
    __device__ __forceinline__ void init(bool go, const uint32_t* c, int bitpos, int regions_old, int path_old) {
        uint32_t po_n = 0, fo_n = 0;
        int mold_n = -1;
        if (go) {
            po_n = c[j];
            fo_n = c[NW + j];
            mold_n = (int)c[2 * NW];
        }
        const uint32_t d = j == (bitpos >> 5) ? 1u << (bitpos & 31) : 0u;
        const uint32_t pn_n = po_n ^ d;
        const bool now_pass = gany(go && (pn_n & d) != 0u);
        const uint32_t seed = nbr(go ? d : 0u) & pn_n;
        if (go) {
            po = po_n;
            fo = fo_n;
            mold = mold_n;
            pn = pn_n;
            regions = regions_old;
            lold = path_old;
            front = now_pass ? d : seed;
            avail = pn & ~front;
            fars = 0;
            unon = 0;
            farrest = 0;
            phase = 0;
            level = 0;
            lu = 0;
            mcu = -1;
            hit = false;
        }
    }
    // LG_EXPAND_R BFS levels of the groups with `run`; returns whether the group's frontier is still alive
    // afterwards (false for !run).  The levels are computed blind, one straight dependent chain of shuffles and
    // logic ops -- a dead frontier stays dead and leaves avail alone, so running past the end is harmless -- and only
    // then the ballots (independent of each other, off the chain) say how many levels were real: front must end up
    // as the LAST NON-EMPTY level (its lowest cell is the far tile) and level counts only those.
    __device__ __forceinline__ bool expand_window(bool run) {
        uint32_t f = front, av = avail, hist[LG_EXPAND_R];
#pragma unroll
        for (int r = 0; r < LG_EXPAND_R; ++r) {
            const uint32_t n = nbr(f) & av;
            av &= ~n;
            f = n;
            hist[r] = n;
        }
        int adv = 0;
        uint32_t last = front;
#pragma unroll
        for (int r = 0; r < LG_EXPAND_R; ++r) {
            const bool some = gany(run && hist[r] != 0u);   // monotone: once a level is empty the later ones are too
            adv += some ? 1 : 0;
            last = some ? hist[r] : last;
        }
        if (run) {
            avail = av;
            front = last;
            level += adv;
        }
        return run && adv == LG_EXPAND_R;
    }
    // The groups with `dead` (busy, frontier died) take their transition; returns true for the groups whose search is
    // over.  Each phase is one block entered by the whole warp if any group needs it.
    __device__ __forceinline__ bool transition(bool dead) {
        bool over = false;
        if (__any_sync(FULL, dead && phase == 0)) {   // flood done: U = P' \ avail
            const bool mine = dead && phase == 0;
            const uint32_t nb = nbr(pn), nbo = nbr(po);
            const uint32_t u = pn & ~avail;
            const uint32_t a = u | (po & ~pn);                   // U | D-
            const int k_old = gsum(__popc(fo & a) + __popc(po & ~nbo & a));
            const uint32_t iso = u & ~nb;
            const int k_iso = gsum(__popc(iso));
            const bool h = gany(mine && mold >= 0 && j == (mold >> 5) && ((a >> (mold & 31)) & 1u));
            if (mine) {
                farrest = fo & ~a;
                hit = h;
                avail = u & ~iso;
                unon = avail;
                front = 0;
                regions += k_iso - k_old;
                phase = 1;
            }
        }
        if (__any_sync(FULL, dead && phase == 1)) {   // first sweeps inside U, one component at a time
            const bool mine = dead && phase == 1;
            uint32_t one_f, one_a;
            lowest(front, &one_f);
            const int nxt = lowest(avail, &one_a);
            const bool more_fars = gany(mine && ((fars | one_f) != 0u));
            if (mine) {
                fars |= one_f;
                if (nxt >= 0) {
                    front = one_a;
                    avail &= ~one_a;
                    ++regions;
                    dead = false;                                // a new first sweep runs
                } else {
                    phase = 2;                                   // joint second sweep inside U
                    front = fars;
                    avail = unon & ~fars;
                    level = 0;
                    if (more_fars) dead = false;
                }
            }
        }
        if (__any_sync(FULL, dead && phase == 2)) {
            const bool mine = dead && phase == 2;
            uint32_t one;
            const int low = lowest(front, &one);
            const bool rest = gany(mine && farrest != 0u);
            if (mine) {
                lu = level;
                mcu = low;
                if (hit) {      // the component that held the maximum was touched: re-sweep the untouched ones
                    front = farrest;
                    avail = pn & ~unon & ~front;                 // isolated cells may stay: never reached
                    phase = 3;
                    level = 0;
                    lold = 0;
                    mold = -1;
                    over = !rest;
                } else {
                    over = true;
                }
                dead = false;
            }
        }
        if (__any_sync(FULL, dead && phase == 3)) {   // the re-sweep died
            uint32_t one;
            const int low = lowest(front, &one);
            if (dead && phase == 3) {
                lold = level;
                mold = low;
                over = true;
            }
        }
        return over;
    }
    __device__ __forceinline__ void finish(int* out, uint32_t* c) const {
        out[0] = regions;
        out[1] = max(lu, lold);
        c[j] = pn;
        c[NW + j] = farrest | fars;
        if (j == 0) c[2 * NW] = (uint32_t)(lu > lold ? mcu : mold);
    }
};

template <int NW>
__global__ void __launch_bounds__(LG_THREADS) k_step_lanegroup(const __grid_constant__ KParams p, const int T) {
    using M = LaneGroupInc<NW>;
    constexpr int WARPS = LG_THREADS / 32;
    constexpr unsigned LEADERS = NW == 8 ? 0x01010101u : NW == 4 ? 0x11111111u : NW == 2 ? 0x55555555u : 0xffffffffu;
    __shared__ int s_cell[WARPS][32];
    __shared__ int2 s_res[WARPS][32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int W = p.d1;
    const int64_t n_warps = (int64_t)gridDim.x * WARPS;
    M m;
    m.lane = lane;
    m.j = lane % NW;
    m.gmask = NW == 32 ? 0xffffffffu : ((1u << NW) - 1u) << (lane - m.j);
    m.pn = m.po = m.fo = m.avail = m.front = m.fars = m.unon = m.farrest = 0;
    m.phase = m.level = m.regions = m.lu = m.lold = 0;
    m.mcu = m.mold = -1;
    m.hit = false;
    const unsigned below = (1u << (lane - m.j)) - 1u;         // the lanes of the groups before mine
    for (int64_t e0 = ((int64_t)blockIdx.x * WARPS + warp) * T; e0 < p.n_envs; e0 += n_warps * T) {
        // ---- update
        const int64_t gid = e0 + lane;
        int cell = -1;
        const bool need = lane < T && gid < p.n_envs && inc_update_env(p, gid, &cell);
        unsigned todo = __ballot_sync(0xffffffffu, need);     // changed envs of the tile not yet handed to a group
        s_cell[warp][lane] = cell;
        __syncwarp();
        // ---- search.  One flat loop, warp-uniform control flow: idle groups take the next changed env, every busy
        // group runs LG_EXPAND_R levels, the groups whose frontier died take their transition.
        bool active = false;
        int slot = 0;
        uint32_t* row = nullptr;
        for (;;) {
            const unsigned idle = __ballot_sync(0xffffffffu, !active) & LEADERS;
            if (todo && idle) {
                const unsigned s = __fns(todo, 0, __popc(idle & below) + 1);
                const bool go = !active && s <= 31u;
                int bitpos = 0, r_old = 0, p_old = 0;
                if (go) {
                    slot = (int)s;
                    const int64_t env = e0 + slot;
                    const int c = s_cell[warp][slot];
                    const int y = c / W, x = c - y * W;
                    bitpos = Board<NW, true>::bitpos(y, x);
                    row = (uint32_t*)(p.cache + env * p.cache_stride);
                    const int2 st = *(const int2*)(p.stats + env * 2);
                    r_old = st.x;
                    p_old = st.y;
                }
                m.init(go, row, bitpos, r_old, p_old);
                active = active || go;
                const int take = min(__popc(idle), __popc(todo));
                const unsigned last = __fns(todo, 0, take);    // position of the last env handed out
                todo &= ~((2u << last) - 1u);
            }
            if (!__any_sync(0xffffffffu, active)) break;
            const bool alive = m.expand_window(active);
            if (m.transition(active && !alive)) {
                int out[2];
                m.finish(out, row);
                if (m.j == 0) s_res[warp][slot] = make_int2(out[0], out[1]);
                active = false;
            }
        }
        __syncwarp();
        // ---- output
        if (need) {
            const int2 r = s_res[warp][lane];
            inc_output_env(p, gid, r.x, r.y);
        }
        __syncwarp();
    }
}

template <int NW>
static cudaError_t launch_lg(const KParams& p, cudaStream_t s) {
    int n_sm = 0;
    const cudaError_t e = sm_count(n_sm);
    if (e != cudaSuccess) return e;
    // tile size: the smallest of 8 / 16 / 32 envs per warp whose grid still fits the GPU in one wave (every warp then
    // runs as few searches one after the other as possible).  At 64 Ki envs, where this picks 16, 8 / 16 / 32 envs per
    // warp gave 0.0810 / 0.0749 / 0.0847 ms per step (profiles/r02_lanegroup_by_size.txt).
    const int64_t resident_warps = (int64_t)n_sm * 32;      // 8 CTAs of 4 warps per SM (64 registers per thread)
    int T = 32;
    if ((p.n_envs + 7) / 8 <= resident_warps) T = 8;
    else if ((p.n_envs + 15) / 16 <= resident_warps) T = 16;
    const int64_t warps = (p.n_envs + T - 1) / T;
    const int64_t want = (warps + LG_THREADS / 32 - 1) / (LG_THREADS / 32);
    const int64_t cap = (int64_t)n_sm * 8;
    k_step_lanegroup<NW><<<(unsigned)(want < cap ? want : cap), LG_THREADS, 0, s>>>(p, T);
    return cudaGetLastError();
}

// MODE_STEP of a binary shard (maps <= 16x16, one-cell edits, per-env search cache present) in one launch
cudaError_t launch_bitboard_lanegroup(const KParams& p, int problem, cudaStream_t s, bool& supported) {
    supported = problem == PCGRL_PROB_BINARY && p.mode == MODE_STEP && p.ndim == 2 && p.d0 <= 16 && p.d1 <= 16 &&
                p.cache != nullptr && p.rep != PCGRL_REP_CELLULAR && p.action_kind != PCGRL_ACT_PATCH;
    if (!supported || p.n_envs == 0) return cudaSuccess;
    return with_board(p.d0, p.d1, supported, [&](auto b) {
        using B = decltype(b);
        if constexpr (!B::TWO_ROWS) return cudaErrorInvalidValue;   // not reached: maps of at most 16x16
        else return launch_lg<B::WORDS>(p, s);
    });
}

}  // namespace pcgrl
