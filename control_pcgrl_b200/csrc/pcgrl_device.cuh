// Shared device-side helpers for the PCGRL step kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include "../../include/pcgrl_b200.h"

namespace pcgrl {

enum { MODE_STEP = 0, MODE_RESET = 1, MODE_STATS = 2 };

// The equivalent step paths of the bit-board problems (binary, zelda, binary_holey), in the order of PCGRL_STEP_PATH's
// names fused | split | inc | incfused | lg:
//   FUSED      k_step_bitboard, one launch (step_bitboard.cu)
//   SPLIT      act / static search / output, three launches over a global work list (step_split.cu)
//   INC        the same with the incremental search from the per-env cache
//   INC_FUSED  the incremental step in one launch, k_step_inc
//   LANEGROUP  k_step_lanegroup, one launch (step_lanegroup.cu)
// A path that does not apply to a shard falls back: lane groups without a search cache run INC_FUSED; INC and INC_FUSED
// without a cache (zelda, binary_holey, maps beyond 16x16) run the static SPLIT; SPLIT on a cellular shard, without a
// work list or on maps beyond 32x32 runs FUSED, and maps beyond 32x32 then run the warp-per-grid boards
// (step_bigboard.cu).
enum StepPath { FUSED, SPLIT, INC, INC_FUSED, LANEGROUP };

// Everything a kernel needs, passed by value (fits the 4 KB parameter space comfortably).
struct KParams {
    int32_t mode;
    int32_t rep, action_kind, ndim;
    int32_t d0, d1, d2;           // numpy axis order; 2D: (H, W, 1)
    int32_t cells, row_stride;
    int32_t n_tiles, n_stats;
    int32_t max_iterations, max_changes;
    int32_t act_h, act_w;
    int32_t targets_per_env;
    int32_t init_random_probs;
    int32_t reward_mode;
    float   init_cdf[PCGRL_MAX_TILES];
    double  weights[PCGRL_MAX_STATS];
    int64_t n_envs, env_offset;
    int8_t* grids;
    int32_t *pos, *n_step, *iteration, *changes, *stats;
    const double* targets;
    float* reward;
    uint8_t *done, *changed;
    int32_t* status;
    void* scratch;
    const void* actions;
    // reset
    const uint8_t* mask;
    const int8_t* src_grids;
    const int32_t* src_pos;
    uint64_t seed, epoch;
    // stats-only mode
    const int8_t* stats_grids;
    int32_t* stats_out;
    // representation wrappers (envs/reps/wrappers.py): action patch, frozen tiles
    int32_t aw0, aw1, aw2;        // MultiActionRepresentation patch size per axis (all 1 when off)
    uint8_t* static_mask;         // [N, row_stride] or NULL
    float   static_prob;
    int32_t n_static_walls, wall_tile, static_eval_mode;
    // holey problems: [N,4] (entrance_y, entrance_x, exit_y, exit_x) in bordered coordinates
    int32_t* holes;
    int32_t hole_mode;
    // compact host I/O (ABI 5): narrow action elements, packed per-env result records
    int32_t act_bytes;            // 4, 1 or 2: element size of PCGRL_ACT_INT32 / PCGRL_ACT_WIDE_FLAT actions
    int32_t rec_stride, rec_sb;   // bytes per record / per stat in it (rec_sb == 0: no records)
    uint8_t* records;             // [N, rec_stride] or NULL
    // split step path (step_split.cu): work list of changed envs + per-env search cache (both may be NULL)
    int32_t* wl_hdr;              // 16 header ints of this launch's work list
    int32_t* worklist;            // its body: [2 ints per env (env, cell) | n_stats ints per env]
    uint8_t* cache;               // [N, cache_stride]
    int32_t cache_stride;
    int32_t host_chunk;           // 1: this launch is one chunk of the host pipeline (other chunks run beside it)
};

// Outputs of one incremental lookahead (lookahead.cu); the KParams beside it have n_envs = the candidate count.
struct LaOut {
    const int32_t* env_idx;   // NULL: candidate j is env j
    int64_t n_src;            // envs of the shard
    float* reward;
    uint8_t* done;
    uint8_t* changed;
    int32_t* stats;
};

// one scalar action (narrow / turtle / flat wide) in the width the caller chose (cfg.action_elem_bytes)
__device__ __forceinline__ int load_action(const KParams& p, int64_t gid) {
    if (p.act_bytes == 1) return ((const uint8_t*)p.actions)[gid];
    if (p.act_bytes == 2) return ((const uint16_t*)p.actions)[gid];
    return ((const int32_t*)p.actions)[gid];
}

// Packed result record of env gid (include/pcgrl_b200.h, pcgrl_state.records):
//   [f32 reward][n_stats x rec_sb bytes][pad][u8 done][u8 changed]
__device__ __forceinline__ void record_flags(const KParams& p, int64_t gid, int done, int changed) {
    if (!p.records) return;
    uint8_t* r = p.records + gid * p.rec_stride;
    *(uint16_t*)(r + p.rec_stride - 2) = (uint16_t)((done ? 1 : 0) | (changed ? 0x100 : 0));
}
__device__ __forceinline__ void record_reward(const KParams& p, int64_t gid, float reward) {
    if (!p.records) return;
    *(float*)(p.records + gid * p.rec_stride) = reward;
}
template <int K>
__device__ __forceinline__ void record_stats(const KParams& p, int64_t gid, const int32_t (&v)[K]) {
    if (!p.records) return;
    uint8_t* r = p.records + gid * p.rec_stride + 4;
    bool fits = true;
    if (p.rec_sb == 1) {
        if (K == 2) {   // binary: both stats in one 16-bit store
            *(uint16_t*)r = (uint16_t)((v[0] & 0xFF) | ((v[1] & 0xFF) << 8));
            fits = ((unsigned)v[0] | (unsigned)v[1]) < 256u;
        } else {
#pragma unroll
            for (int k = 0; k < K; ++k) {
                r[k] = (uint8_t)v[k];
                fits = fits && (unsigned)v[k] < 256u;
            }
        }
    } else if (p.rec_sb == 2) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            ((int16_t*)r)[k] = (int16_t)v[k];
            fits = fits && v[k] == (int)(int16_t)v[k];
        }
    } else {
#pragma unroll
        for (int k = 0; k < K; ++k) ((int32_t*)r)[k] = v[k];
    }
    if (!fits && p.status) atomicOr(p.status, 16);
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), counter-based: no RNG state lives in HBM.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

// ------------------------------------------------------------------------------------------------
// ControlWrapper.get_loss (control_wrappers.py:318-345) for one env, in fp64 from integer stats.
//   scalar target:  -|trg - val| * w
//   range (lo,hi):  -min_j |lo + j - val| * w   over j = 0 .. ceil(hi-lo)-1   (np.arange(lo,hi), hi excluded)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double control_loss(const int32_t* st, const double* trg, const double* w, int K) {
    double loss = 0.0;
    for (int k = 0; k < K; ++k) {
        const double wk = w[k];
        if (wk == 0.0) continue;
        const double lo = trg[2 * k], hi = trg[2 * k + 1], v = (double)st[k];
        double d;
        if (isnan(hi)) {
            d = fabs(lo - v);
        } else {
            const double n = ceil(hi - lo);
            double j = rint(v - lo);
            j = fmin(fmax(j, 0.0), n - 1.0);
            d = fabs(lo + j - v);
        }
        loss += -d * wk;
    }
    return loss;
}

// ------------------------------------------------------------------------------------------------
// Legacy Problem.get_reward: sum_k w_k * get_range_reward(new_k, old_k, lo_k, hi_k)  (envs/helper.py:550-560;
// the bands may be +-infinity, e.g. "the longer the better" = (inf, inf), binary_prob.py:170-178).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double range_reward(double nv, double ov, double lo, double hi) {
    if (nv >= lo && nv <= hi && ov >= lo && ov <= hi) return 0.0;
    if (ov <= hi && nv <= hi) return fmin(nv, lo) - fmin(ov, lo);
    if (ov >= lo && nv >= lo) return fmax(ov, hi) - fmax(nv, hi);
    if (nv > hi && ov < lo) return hi - nv + ov - lo;
    if (nv < lo && ov > hi) return hi - ov + nv - lo;
    return 0.0;   // unreachable for lo <= hi (the reference would return None)
}
__device__ __forceinline__ double range_reward_sum(const int32_t* nw, const int32_t* od, const double* band,
                                                   const double* w, int K) {
    double r = 0.0;
    for (int k = 0; k < K; ++k)
        if (w[k] != 0.0) r += w[k] * range_reward((double)nw[k], (double)od[k], band[2 * k], band[2 * k + 1]);
    return r;
}

// ------------------------------------------------------------------------------------------------
// Bit-boards: one thread owns one level grid as NW 32-bit words held in registers.
//   TWO = true : a word holds two rows of up to 16 cells (row 2i in bits 0..15, row 2i+1 in 16..31)
//   TWO = false: a word holds one row of up to 32 cells
// Bit order (word, bit) is monotonic in the row-major cell index, so "lowest set bit of the board"
// == "first cell in the reference's y-outer/x-inner scan" (envs/helper.py:23-25).
// No cross-lane traffic at all: x+-1 are shifts inside a word, y+-1 are funnel shifts between
// neighbouring words (TWO) or plain neighbouring words.
// ------------------------------------------------------------------------------------------------
template <int NW, bool TWO>
struct Board {
    static constexpr int WORDS = NW;
    static constexpr bool TWO_ROWS = TWO;
    // bit position (word * 32 + bit) of cell (y, x)
    __host__ __device__ static constexpr int bitpos(int y, int x) { return TWO ? y * 16 + x : y * 32 + x; }
    // n = dilate4(f) & av;  returns OR of all words of n (zero <=> frontier died)
    //
    // TWO layout: the "row above" word of board word i and the "row below" word of board word i-1 are the
    // same 32-bit window straddling words i-1 and i (high row of i-1, low row of i), so one funnel shift
    // per word boundary serves both directions.  x<<1 is an add (IMAD.IADD, FMA pipe).  x>>1 and the 16-bit funnel
    // shifts stay SHF on the ALU pipe: issuing them as IMAD.HI was SLOWER on B200, 0.2997 ms per step against 0.3064
    // (shr), 0.3092 (funnel), 0.3225 (both) at 1 Mi envs -- IMAD.HI is not a full-rate instruction.
    __device__ static __forceinline__ uint32_t expand_and(const uint32_t (&f)[NW], const uint32_t (&av)[NW],
                                                          uint32_t (&n)[NW]) {
        uint32_t any = 0;
        if (TWO) {
            uint32_t s[NW + 1];  // s[i] = rows (2i-1, 2i): window between word i-1 and word i
            s[0] = f[0] << 16;
#pragma unroll
            for (int i = 1; i < NW; ++i) s[i] = __funnelshift_l(f[i - 1], f[i], 16);
            s[NW] = f[NW - 1] >> 16;
#pragma unroll
            for (int i = 0; i < NW; ++i) {
                // the two 16-bit rows of a word must not leak into each other.  Rows narrower than 16 have
                // never-passable padding bits, for which the masks are no-ops, so they are always applied.
                const uint32_t l = (f[i] + f[i]) & 0xFFFEFFFEu;
                const uint32_t r = (f[i] >> 1) & 0x7FFF7FFFu;
                n[i] = (l | r | s[i] | s[i + 1]) & av[i];
                any |= n[i];
            }
        } else {
#pragma unroll
            for (int i = 0; i < NW; ++i) {
                const uint32_t up = i > 0 ? f[i - 1] : 0u;
                const uint32_t dn = i < NW - 1 ? f[i + 1] : 0u;
                n[i] = ((f[i] + f[i]) | (f[i] >> 1) | up | dn) & av[i];
                any |= n[i];
            }
        }
        return any;
    }
    // t = x - 1 as one multi-word integer (borrow rippling up through sub.cc / subc.cc); returns true iff x != 0.
    // With it the lowest set cell of x is x & ~t and x without that cell is x & t -- one LOP3 per word each, which
    // ptxas fuses with the consumer (fars |= x & ~t), instead of a negate / and / xor sequence (X & -X).
    __device__ static __forceinline__ bool minus_one(const uint32_t (&x)[NW], uint32_t (&t)[NW]) {
        uint32_t b;
        if constexpr (NW == 1) {
            t[0] = x[0] - 1u;
            return x[0] != 0u;
        } else if constexpr (NW == 2) {
            asm("sub.cc.u32 %0, %3, 1;\n\tsubc.cc.u32 %1, %4, 0;\n\tsubc.u32 %2, 0, 0;"
                : "=r"(t[0]), "=r"(t[1]), "=r"(b) : "r"(x[0]), "r"(x[1]));
            return b == 0u;
        } else if constexpr (NW == 4) {
            asm("sub.cc.u32 %0, %5, 1;\n\tsubc.cc.u32 %1, %6, 0;\n\tsubc.cc.u32 %2, %7, 0;\n\tsubc.cc.u32 %3, %8, 0;\n\t"
                "subc.u32 %4, 0, 0;"
                : "=r"(t[0]), "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(b)
                : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(x[3]));
            return b == 0u;
        } else if constexpr (NW == 8) {
            asm("sub.cc.u32 %0, %9, 1;\n\tsubc.cc.u32 %1, %10, 0;\n\tsubc.cc.u32 %2, %11, 0;\n\t"
                "subc.cc.u32 %3, %12, 0;\n\tsubc.cc.u32 %4, %13, 0;\n\tsubc.cc.u32 %5, %14, 0;\n\t"
                "subc.cc.u32 %6, %15, 0;\n\tsubc.cc.u32 %7, %16, 0;\n\tsubc.u32 %8, 0, 0;"
                : "=r"(t[0]), "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7]), "=r"(b)
                : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(x[3]), "r"(x[4]), "r"(x[5]), "r"(x[6]), "r"(x[7]));
            return b == 0u;
        } else {
            uint32_t borrow = 1, nz = 0;
#pragma unroll
            for (int i = 0; i < NW; ++i) {
                t[i] = x[i] - borrow;
                borrow = (x[i] < borrow) ? 1u : 0u;
                nz |= x[i];
            }
            return nz != 0u;
        }
    }
    // x \ n for n a subset of x, as x - n: an IMAD on the FMA pipe instead of a LOP3 on the (saturated) ALU pipe
    __device__ static __forceinline__ uint32_t minus_subset(uint32_t x, uint32_t n) {
        uint32_t r;
        asm("mad.lo.u32 %0, %1, 0xFFFFFFFF, %2;" : "=r"(r) : "r"(n), "r"(x));
        return r;
    }
    __device__ static __forceinline__ uint32_t any(const uint32_t (&x)[NW]) {
        uint32_t r = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) r |= x[i];
        return r;
    }
    __device__ static __forceinline__ int popcount(const uint32_t (&x)[NW]) {
        int c = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) c += __popc(x[i]);
        return c;
    }
    __device__ static __forceinline__ uint32_t any_and(const uint32_t (&a)[NW], const uint32_t (&b)[NW]) {
        uint32_t r = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) r |= a[i] & b[i];
        return r;
    }
};

// The board of a d0 x d1 map (rows x columns): up to 16x16 two rows per word in 1 / 2 / 4 / 8 words, up to 32x32 one
// row per word in 16 / 32 words.  Returns f(Board<NW, TWO>{}); a larger map has no board: supported = false and f is
// not called.
template <class F>
auto with_board(int d0, int d1, bool& supported, F&& f) -> decltype(f(Board<1, true>{})) {
    supported = true;
    if (d1 <= 16 && d0 <= 16) {
        const int nw = (d0 + 1) / 2;
        if (nw <= 1) return f(Board<1, true>{});
        if (nw <= 2) return f(Board<2, true>{});
        if (nw <= 4) return f(Board<4, true>{});
        return f(Board<8, true>{});
    }
    if (d1 <= 32 && d0 <= 32) {
        if (d0 <= 16) return f(Board<16, false>{});
        return f(Board<32, false>{});
    }
    supported = false;
    return {};
}

// SM count of the current device, queried once per device (ordinals beyond 16 on every call)
inline cudaError_t sm_count(int& n) {
    static std::atomic<int> cached[16];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const bool slot = dev >= 0 && dev < 16;
    if (slot && (n = cached[dev].load(std::memory_order_relaxed)) > 0) return cudaSuccess;
    if ((e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    if (slot) cached[dev].store(n, std::memory_order_relaxed);
    return cudaSuccess;
}

}  // namespace pcgrl
