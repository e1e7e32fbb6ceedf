// Skeleton of the warp-per-grid step kernels (problems whose get_stats is an order-dependent sequential
// search: minecraft_3D_maze, sokoban, smb).  Same phases as the bit-board kernel (step_bitboard.cu), but
//   - the grid of CTAs is persistent (one or more CTAs per SM looping over tiles of TILE envs), so that the
//     per-warp search workspaces (shared memory, plus global scratch for the big node pools) are bounded by
//     the number of resident warps, not by the number of envs;
//   - phase C hands each changed env to a whole warp: lane-parallel where the work is data-parallel (grid
//     load, bit-board construction, flood fill, child generation), warp-uniform where the reference's
//     queue order has to be reproduced step by step.
#pragma once
#include <atomic>
#include "pcgrl_device.cuh"
#include "step_common.cuh"

namespace pcgrl {

constexpr int SEARCH_WARPS = 8;   // default warps per CTA (a problem may ask for more)
constexpr int SEARCH_TILE = 64;                  // envs per CTA iteration (a CTA-wide barrier closes each one).  A/B on the 3D
                                                 // maze (65 536 envs): 32 / 64 / 128 / 256 -> 2.19 / 2.25 / 2.18 / 1.41e7 env-steps/s
constexpr int SEARCH_SLOTS = 64;  // concurrent launches that can share the tile counters below
// Dynamic tile scheduling: CTAs pull tile indices from g_tile_ctr[slot]; the last CTA to leave resets the
// slot, so nothing has to be zeroed from the host between launches.  The host hands out slots round-robin.
static __device__ unsigned int g_tile_ctr[SEARCH_SLOTS];
static __device__ unsigned int g_done_ctr[SEARCH_SLOTS];
constexpr int SEARCH_MAX_CTAS = 320;   // persistent-grid cap that sizes the global scratch (>= 2 CTAs x 148 SMs)

// floor(n / d) for n < 2^16 and d <= 2^8 as one multiply-high: magic = ceil(2^32 / d)
__host__ __device__ inline uint32_t div_magic(int d) { return (uint32_t)((0x100000000ull + d - 1) / d); }
__device__ __forceinline__ int div_by(int n, uint32_t magic) { return magic ? (int)__umulhi((uint32_t)n, magic) : n; }  // magic == 0 <=> d == 1

// ------------------------------------------------------------------------------------------------
// calc_num_regions (helper.py:200-210 / helper_3D.py:396-406) as connected-component labelling with a
// shared-memory union-find over *runs*: rows[z * Y + y] is the bit mask over x of passable cells; a run is
// a maximal horizontal stretch of set bits, identified by the cell index of its first cell.  Every run is
// united with the runs it touches in the row above (y - 1) and in the plane below (z - 1); the number of
// regions is the number of roots.  6-neighbour in 3D, 4-neighbour when Z == 1.  Whole warp, lanes stride
// the rows; parent[] needs Z*Y*X u16 entries.  Lock-free: the larger root is hooked under the smaller one
// with a 16-bit compare-and-swap and retried on interference.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int run_start(uint32_t a, int b) {
    const uint32_t below = ~a & ((1u << b) - 1u);     // zero bits under b
    return 32 - __clz(below);                         // first bit of the run that contains b
}
__device__ inline void uf_union(volatile uint16_t* parent, int a, int b) {
    for (;;) {
        int pa, pb;
        // find with path halving: every visited node is re-pointed at its grandparent.  Racing lanes only ever
        // replace a pointer by another ancestor of the same node, so the forest stays valid without locks.
        while ((pa = parent[a]) != a) {
            const int ga = parent[pa];
            if (ga != pa) parent[a] = (uint16_t)ga;
            a = ga;
        }
        while ((pb = parent[b]) != b) {
            const int gb = parent[pb];
            if (gb != pb) parent[b] = (uint16_t)gb;
            b = gb;
        }
        if (a == b) return;
        if (a < b) {
            const int t = a;
            a = b;
            b = t;
        }
        const unsigned short old = atomicCAS((unsigned short*)parent + a, (unsigned short)a, (unsigned short)b);
        if (old == (unsigned short)a) return;
    }
}
__device__ inline int count_regions_rows(const uint16_t* row, int Z, int Y, int X, uint16_t* parent, int lane) {
    const int R = Z * Y;
    const uint32_t magic_y = div_magic(Y);
    for (int r = lane; r < R; r += 32) {
        const uint32_t a = row[r];
        for (uint32_t s = a & ~(a << 1); s; s &= s - 1) {
            const int id = r * X + __ffs(s) - 1;
            parent[id] = (uint16_t)id;
        }
    }
    __syncwarp();
    for (int r = lane; r < R; r += 32) {
        const int z = div_by(r, magic_y), y = r - z * Y;
        const uint32_t a = row[r];
        if (!a) continue;
#pragma unroll
        for (int dir = 0; dir < 2; ++dir) {
            if (dir == 0 ? y == 0 : z == 0) continue;
            const int rp = dir == 0 ? r - 1 : r - Y;
            const uint32_t ap = row[rp];
            const uint32_t t = a & ap;                          // vertically adjacent passable pairs
            for (uint32_t s = t & ~(t << 1); s; s &= s - 1) {   // one union per stretch of such pairs
                const int bpos = __ffs(s) - 1;
                uf_union(parent, r * X + run_start(a, bpos), rp * X + run_start(ap, bpos));
            }
        }
    }
    __syncwarp();
    int roots = 0;
    for (int r = lane; r < R; r += 32) {
        const uint32_t a = row[r];
        for (uint32_t s = a & ~(a << 1); s; s &= s - 1) {
            const int id = r * X + __ffs(s) - 1;
            roots += parent[id] == id;
        }
    }
    return __reduce_add_sync(0xffffffffu, roots);
}

// The same labelling with 32-bit parents indexed by (row, k-th run of the row): rows are at most 16 cells wide, so a
// row has at most 8 runs and `parent` needs Z*Y*8 words -- about the size of the per-cell u16 table for 14-wide
// rows, but the hook is a native 32-bit atomicCAS instead of the 16-bit one CUDA emulates with a CAS loop on the
// containing word.
__device__ __forceinline__ int run_id(uint32_t a, int r, int bpos) {
    const uint32_t starts = a & ~(a << 1);
    return r * 8 + __popc(starts & ((2u << bpos) - 1u)) - 1;   // bpos lies in its run, at or above the run's start
}
__device__ inline void uf_union32(volatile uint32_t* parent, int a, int b) {
    for (;;) {
        int pa, pb;
        while ((pa = (int)parent[a]) != a) {
            const int ga = (int)parent[pa];
            if (ga != pa) parent[a] = (uint32_t)ga;
            a = ga;
        }
        while ((pb = (int)parent[b]) != b) {
            const int gb = (int)parent[pb];
            if (gb != pb) parent[b] = (uint32_t)gb;
            b = gb;
        }
        if (a == b) return;
        if (a < b) {
            const int t = a;
            a = b;
            b = t;
        }
        if (atomicCAS((unsigned int*)parent + a, (unsigned int)a, (unsigned int)b) == (unsigned int)a) return;
    }
}
__device__ inline int count_regions_runs32(const uint16_t* row, int Z, int Y, int X, uint32_t* parent, int lane) {
    const int R = Z * Y;
    const uint32_t magic_y = div_magic(Y);
    for (int r = lane; r < R; r += 32) {
        const uint32_t a = row[r];
        const int n = __popc(a & ~(a << 1));
        for (int k = 0; k < n; ++k) parent[r * 8 + k] = (uint32_t)(r * 8 + k);
    }
    __syncwarp();
    for (int r = lane; r < R; r += 32) {
        const int z = div_by(r, magic_y), y = r - z * Y;
        const uint32_t a = row[r];
        if (!a) continue;
#pragma unroll
        for (int dir = 0; dir < 2; ++dir) {
            if (dir == 0 ? y == 0 : z == 0) continue;
            const int rp = dir == 0 ? r - 1 : r - Y;
            const uint32_t ap = row[rp];
            const uint32_t t = a & ap;                          // vertically adjacent passable pairs
            for (uint32_t s = t & ~(t << 1); s; s &= s - 1) {   // one union per stretch of such pairs
                const int bpos = __ffs(s) - 1;
                uf_union32(parent, run_id(a, r, bpos), run_id(ap, rp, bpos));
            }
        }
    }
    __syncwarp();
    int roots = 0;
    for (int r = lane; r < R; r += 32) {
        const uint32_t a = row[r];
        const int n = __popc(a & ~(a << 1));
        for (int k = 0; k < n; ++k) roots += parent[r * 8 + k] == (uint32_t)(r * 8 + k);
    }
    return __reduce_add_sync(0xffffffffu, roots);
}

// Prob must provide:
//   static constexpr int K;
//   struct Ctx;                                         per-warp context (pointers into its workspaces)
//   static __device__ Ctx make_ctx(const KParams&, uint8_t* warp_smem, int global_warp);
//   static __device__ void stats(const KParams&, Ctx&, const int8_t* grid, int lane, int32_t* out /*smem [K]*/);
template <class Prob, int WARPS>
__global__ void __launch_bounds__(WARPS * 32) k_step_search(const KParams p, const int smem_per_warp, const int slot,
                                                             const int64_t tile_begin, const int64_t tile_end) {
    constexpr int K = Prob::K;
    constexpr int TILE = SEARCH_TILE;
    constexpr int SEARCH_THREADS = WARPS * 32;
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    __shared__ int32_t s_stats[TILE * K];
    __shared__ int16_t s_list[TILE];
    __shared__ int16_t s_slot[TILE];
    __shared__ uint8_t s_flag[TILE];
    __shared__ int s_count, s_next;
    __shared__ unsigned int s_tile;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int8_t* grids_in = (p.mode == MODE_STATS) ? p.stats_grids : p.grids;
    typename Prob::Ctx ctx = Prob::make_ctx(p, dyn_smem + (size_t)warp * smem_per_warp, blockIdx.x * WARPS + warp);
    for (;;) {
        __syncthreads();   // previous tile's phase D is done with the shared lists
        if (tid == 0) {
            s_tile = atomicAdd(&g_tile_ctr[slot], 1u);
            s_count = 0;
            s_next = 0;
        }
        __syncthreads();
        const int64_t tile = tile_begin + s_tile;   // this launch covers tiles [tile_begin, tile_end)
        if (tile >= tile_end) break;
        const int64_t base = tile * TILE;
        const int tile_n = (int)min((int64_t)TILE, p.n_envs - base);
        for (int e = tid; e < TILE; e += SEARCH_THREADS) {
            s_slot[e] = -1;
            s_flag[e] = 0;
        }
        __syncthreads();
        phase_a<SEARCH_THREADS, TILE>(p, base, tile_n, s_list, s_slot, s_flag, &s_count);
        const int M = s_count;

        // phase C: one warp per changed env, pulled from the shared queue
        for (;;) {
            int item = 0;
            if (lane == 0) item = atomicAdd(&s_next, 1);
            item = __shfl_sync(0xffffffffu, item, 0);
            if (item >= M) break;
            const int8_t* grid = grids_in + (base + s_list[item]) * p.row_stride;
            Prob::stats(p, ctx, grid, lane, s_stats + item * K);
            __syncwarp();
        }
        __syncthreads();
        phase_d<SEARCH_THREADS, K>(p, base, tile_n, s_slot, s_stats);
    }
    if (tid == 0) {   // last CTA out re-arms the counters for the next launch that gets this slot
        __threadfence();
        if (atomicAdd(&g_done_ctr[slot], 1u) == gridDim.x - 1) {
            g_tile_ctr[slot] = 0;
            g_done_ctr[slot] = 0;
            __threadfence();
        }
    }
}

// host side: persistent launch sized from the occupancy the dynamic shared memory allows
template <class Prob, int WARPS = SEARCH_WARPS>
static cudaError_t launch_search(const KParams& p, cudaStream_t s, int smem_per_warp, int max_ctas_per_sm = 1 << 20,
                                 int max_ctas = SEARCH_MAX_CTAS, int64_t env_begin = 0, int64_t env_end = -1) {
    static std::atomic<unsigned> next_slot{0};
    constexpr int SEARCH_THREADS = WARPS * 32;
    int n_sm = 0;
    cudaError_t e;
    if ((e = sm_count(n_sm)) != cudaSuccess) return e;
    const int dyn = smem_per_warp * WARPS;
    auto kern = k_step_search<Prob, WARPS>;
    if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn)) != cudaSuccess) return e;
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SEARCH_THREADS, dyn)) != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    // envs [env_begin, env_end) only (whole tiles; default: the whole shard) -- for problems that bound the work of a launch
    if (env_end < 0 || env_end > p.n_envs) env_end = p.n_envs;
    const int64_t tile_begin = env_begin / SEARCH_TILE, tile_end = (env_end + SEARCH_TILE - 1) / SEARCH_TILE;
    const int64_t tiles = tile_end - tile_begin;
    if (tiles <= 0) return cudaSuccess;
    if (per_sm > max_ctas_per_sm) per_sm = max_ctas_per_sm;
    int64_t cap = (int64_t)n_sm * per_sm;
    if (max_ctas_per_sm < (1 << 20) && cap > max_ctas) cap = max_ctas;   // the global scratch is sized for this
    const int ctas = (int)(tiles < cap ? tiles : cap);
    const int slot = (int)(next_slot.fetch_add(1) % SEARCH_SLOTS);
    kern<<<ctas, SEARCH_THREADS, dyn, s>>>(p, smem_per_warp, slot, tile_begin, tile_end);
    return cudaGetLastError();
}

}  // namespace pcgrl
