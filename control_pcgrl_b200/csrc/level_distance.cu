// Level distances (pcgrl_level_distances / pcgrl_level_knn / pcgrl_level_group_diversity): d(a, b) is the number of
// the first `cells` bytes (tile codes) in which two levels differ.
//   k_ld_pack    tile codes -> P bit-planes of `cells` bits padded to 32-bit words, one warp per (level, word): lane l
//                reads cell 32 w + l (nothing past `cells`, so the tail bits are 0 on both sides and row padding never
//                counts), then one ballot per plane.  Then d(a, b) = sum_w popc(OR_p a_p[w] ^ b_p[w]).
//   k_ld_tile    32 queries x 128 archive levels per trip, both staged in shared memory with an odd word pitch (lanes
//                read consecutive levels from distinct banks).  Warp v owns queries 4v .. 4v + 3 and lane l the archive
//                levels l, l + 32, l + 64, l + 96 of the trip: 16 pairs per thread, each shared word used 4 times.
//                FULL stores the int32 distances.  Otherwise each warp keeps, per query, the k smallest 64-bit keys
//                (d << 32 | archive index) as a sorted list in registers (lane l holds ranks l and l + 32), so equal
//                distances go to the lower index; a candidate is compared with rank k - 1 and the few that pass are
//                inserted one at a time by the whole warp.  The distance matrix is never written.
//                blockIdx.y is an archive slice: with one slice the lists go straight to the output, otherwise to
//                `work` for k_ld_merge.
//   k_ld_merge   one warp per query runs the same insertion over the slices' lists.
//   k_ld_groups  one block per group of S levels, one unordered pair per thread and trip, int64 block sum.
#include "level_distance.cuh"

namespace pcgrl {

constexpr int LD_THREADS = 256, LD_QT = 32, LD_BT = 128;   // 8 warps x 4 queries; 4 archive levels per lane
constexpr int LD_GROUP_THREADS = 128;
constexpr int LD_MAX_SLICES = 64;
constexpr int LD_SMEM_MAX = 227 * 1024;
constexpr uint64_t LD_NONE = ~0ull;      // no candidate: sorts after every real key, read back as (-1, -1)
constexpr unsigned FULL_MASK = 0xffffffffu;

LdGeom ld_geom(int cells, int n_tiles) {
    LdGeom g;
    g.cells = cells;
    g.W = (cells + 31) / 32;
    g.P = 1;
    while ((1 << g.P) < n_tiles) ++g.P;
    g.L = g.W * g.P;
    return g;
}

static int ld_pitch(const LdGeom& g) { return g.L | 1; }
static size_t ld_tile_smem(const LdGeom& g) { return (size_t)(LD_QT + LD_BT) * ld_pitch(g) * sizeof(uint32_t); }
bool ld_fits(const LdGeom& g) { return ld_tile_smem(g) <= (size_t)LD_SMEM_MAX; }

static int64_t align256(int64_t x) { return (x + 255) / 256 * 256; }

// Archive slices of a kNN call, from the shapes alone: enough blocks to fill the GPU several times over when the
// queries alone do not (1 Ki queries are only 32 blocks), yet at least 8 trips per slice, so that the merge reads few
// lists per query.
struct LdSplit {
    int64_t slices, slice_len;
};
static LdSplit ld_split(int64_t n_q, int64_t n_b) {
    const int64_t q_blocks = (n_q + LD_QT - 1) / LD_QT, trips = (n_b + LD_BT - 1) / LD_BT;
    int64_t s = (1024 + q_blocks - 1) / q_blocks;
    s = s < trips / 8 ? s : trips / 8;
    s = s < LD_MAX_SLICES ? s : LD_MAX_SLICES;
    if (s < 1) s = 1;
    LdSplit r;
    r.slice_len = (trips + s - 1) / s * LD_BT;
    r.slices = r.slice_len ? (n_b + r.slice_len - 1) / r.slice_len : 1;
    if (r.slices < 1) r.slices = 1;
    return r;
}

int64_t ld_work_bytes(const LdGeom& g, int64_t n_a, int64_t n_b, int k) {
    int64_t bytes = align256(n_a * g.L * 4) + align256(n_b * g.L * 4);
    if (k > 0) {
        const LdSplit sp = ld_split(n_a, n_b);
        if (sp.slices > 1) bytes += sp.slices * n_a * k * 8;
    }
    return bytes;
}

__global__ void k_ld_pack(const uint8_t* __restrict__ src, int64_t n, int64_t stride, int cells, int W, int P,
                          uint32_t* __restrict__ dst) {
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // (level, word), warp-uniform
    const int lane = threadIdx.x & 31;
    if (gw >= n * W) return;
    const int64_t lv = gw / W;
    const int w = (int)(gw - lv * W), c = 32 * w + lane;
    const unsigned v = c < cells ? src[lv * stride + c] : 0u;
    uint32_t mine = 0;
    for (int p = 0; p < P; ++p) {
        const uint32_t b = __ballot_sync(FULL_MASK, (v >> p) & 1u);
        if (lane == p) mine = b;
    }
    if (lane < P) dst[gw * P + lane] = mine;
}

// Inserts x (smaller than rank k - 1) into the warp's sorted list: lane l holds ranks l (r0) and l + 32 (r1).
__device__ __forceinline__ void ld_insert(uint64_t& r0, uint64_t& r1, uint64_t x, int lane) {
    const int pos = __popc(__ballot_sync(FULL_MASK, r0 < x)) + __popc(__ballot_sync(FULL_MASK, r1 < x));
    const uint64_t up0 = __shfl_up_sync(FULL_MASK, r0, 1);   // rank lane - 1
    uint64_t up1 = __shfl_up_sync(FULL_MASK, r1, 1);         // rank lane + 31
    const uint64_t last0 = __shfl_sync(FULL_MASK, r0, 31);   // rank 31
    if (lane == 0) up1 = last0;
    r0 = lane < pos ? r0 : lane == pos ? x : up0;
    r1 = lane + 32 < pos ? r1 : lane + 32 == pos ? x : up1;
}

__device__ __forceinline__ uint64_t ld_kth(uint64_t r0, uint64_t r1, int k) {
    return __shfl_sync(FULL_MASK, k <= 32 ? r0 : r1, (k - 1) & 31);
}

// Offers every lane's candidate c to the list; thr is rank k - 1 before and after.
__device__ __forceinline__ void ld_offer(uint64_t& r0, uint64_t& r1, uint64_t& thr, uint64_t c, int k, int lane) {
    unsigned m = __ballot_sync(FULL_MASK, c < thr);
    while (m) {
        const uint64_t x = __shfl_sync(FULL_MASK, c, __ffs(m) - 1);
        m &= m - 1;
        if (x < thr) {   // warp-uniform
            ld_insert(r0, r1, x, lane);
            thr = ld_kth(r0, r1, k);
        }
    }
}

__device__ __forceinline__ void ld_write_list(uint64_t r0, uint64_t r1, int k, int lane, int32_t* dist, int32_t* idx) {
    if (lane < k) {
        dist[lane] = r0 == LD_NONE ? -1 : (int32_t)(r0 >> 32);
        idx[lane] = r0 == LD_NONE ? -1 : (int32_t)(uint32_t)r0;
    }
    if (lane + 32 < k) {
        dist[lane + 32] = r1 == LD_NONE ? -1 : (int32_t)(r1 >> 32);
        idx[lane + 32] = r1 == LD_NONE ? -1 : (int32_t)(uint32_t)r1;
    }
}

struct LdTile {
    const uint32_t* qa;   // packed queries [n_q, L]
    const uint32_t* ba;   // packed archive [n_b, L]
    int64_t n_q, n_b;
    int L, pitch;
    int64_t slice_len;
    int k;
    int64_t self_offset;  // query i is archive level i + self_offset; < 0: none
    int32_t* out;         // FULL: [n_q, n_b]; kNN with one slice: distances [n_q, k]
    int32_t* out_idx;     // kNN with one slice: indices [n_q, k]
    uint64_t* partial;    // kNN with several slices: [slices, n_q, k] keys
};

template <int P, bool FULL>
__global__ void __launch_bounds__(LD_THREADS) k_ld_tile(const LdTile a) {
    extern __shared__ uint32_t ld_smem[];
    uint32_t* sq = ld_smem;
    uint32_t* sb = ld_smem + LD_QT * a.pitch;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t q0 = (int64_t)blockIdx.x * LD_QT;
    const int L = a.L, pitch = a.pitch;
    for (int i = threadIdx.x; i < LD_QT * L; i += LD_THREADS) {
        const int r = i / L;
        sq[r * pitch + (i - r * L)] = q0 + r < a.n_q ? a.qa[q0 * L + i] : 0u;
    }
    const int64_t b_lo = (int64_t)blockIdx.y * a.slice_len;
    const int64_t b_hi = b_lo + a.slice_len < a.n_b ? b_lo + a.slice_len : a.n_b;
    uint64_t r0[4], r1[4], thr[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) r0[i] = r1[i] = thr[i] = LD_NONE;
    const uint32_t* qrow = sq + warp * 4 * pitch;
    for (int64_t t0 = b_lo; t0 < b_hi; t0 += LD_BT) {
        __syncthreads();   // the queries are staged / the previous trip's levels are consumed
        const int nb = b_hi - t0 < LD_BT ? (int)(b_hi - t0) : LD_BT;
        const uint32_t* g = a.ba + t0 * L;
        for (int i = threadIdx.x; i < nb * L; i += LD_THREADS) {
            const int r = i / L;
            sb[r * pitch + (i - r * L)] = g[i];
        }
        __syncthreads();
        int acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0;
        const uint32_t* brow = sb + lane * pitch;
        for (int w = 0; w < L; w += P) {
            uint32_t x[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) x[i][j] = 0;
#pragma unroll
            for (int p = 0; p < P; ++p) {
                uint32_t bv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) bv[j] = brow[32 * j * pitch + w + p];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t qv = qrow[i * pitch + w + p];
#pragma unroll
                    for (int j = 0; j < 4; ++j) x[i][j] |= qv ^ bv[j];
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] += __popc(x[i][j]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t q = q0 + warp * 4 + i;
            if (q >= a.n_q) break;   // warp-uniform
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int64_t b = t0 + lane + 32 * j;
                if constexpr (FULL) {
                    if (b < b_hi) a.out[q * a.n_b + b] = acc[i][j];
                } else {
                    const bool ok = b < b_hi && (a.self_offset < 0 || b != q + a.self_offset);
                    const uint64_t c = ok ? ((uint64_t)(uint32_t)acc[i][j] << 32) | (uint64_t)b : LD_NONE;
                    ld_offer(r0[i], r1[i], thr[i], c, a.k, lane);
                }
            }
        }
    }
    if constexpr (!FULL) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t q = q0 + warp * 4 + i;
            if (q >= a.n_q) break;
            if (a.partial) {
                uint64_t* dst = a.partial + ((int64_t)blockIdx.y * a.n_q + q) * a.k;
                if (lane < a.k) dst[lane] = r0[i];
                if (lane + 32 < a.k) dst[lane + 32] = r1[i];
            } else {
                ld_write_list(r0[i], r1[i], a.k, lane, a.out + q * a.k, a.out_idx + q * a.k);
            }
        }
    }
}

__global__ void k_ld_merge(const uint64_t* __restrict__ partial, int64_t n_q, int64_t slices, int k, int32_t* dist,
                           int32_t* idx) {
    const int64_t q = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q >= n_q) return;   // warp-uniform
    uint64_t r0 = LD_NONE, r1 = LD_NONE, thr = LD_NONE;
    for (int64_t s = 0; s < slices; ++s) {
        const uint64_t* src = partial + (s * n_q + q) * k;
        for (int c = 0; c < k; c += 32) {
            const uint64_t x = c + lane < k ? src[c + lane] : LD_NONE;
            ld_offer(r0, r1, thr, x, k, lane);
        }
    }
    ld_write_list(r0, r1, k, lane, dist + q * k, idx + q * k);
}

template <int P>
__device__ __forceinline__ int ld_dist(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, int L) {
    int d = 0;
    for (int w = 0; w < L; w += P) {
        uint32_t x = 0;
#pragma unroll
        for (int p = 0; p < P; ++p) x |= __ldg(a + w + p) ^ __ldg(b + w + p);
        d += __popc(x);
    }
    return d;
}

// Unordered pairs of a group, without waste: pair t < S h (h = (S - 1) / 2) is (i, (i + 1 + t % h) % S) with
// i = t / h, i.e. every level with the h levels after it around the circle; for even S the S / 2 pairs (i, i + S / 2),
// i < S / 2, follow.
template <int P>
__global__ void __launch_bounds__(LD_GROUP_THREADS) k_ld_groups(const uint32_t* __restrict__ pk, int L, int64_t S,
                                                                 int64_t* __restrict__ sums) {
    const uint32_t* base = pk + (int64_t)blockIdx.x * S * L;
    const int64_t h = (S - 1) / 2, n_pairs = S * (S - 1) / 2;
    int64_t sum = 0;
    for (int64_t t = threadIdx.x; t < n_pairs; t += LD_GROUP_THREADS) {
        int64_t i, j;
        if (t < S * h) {
            i = t / h;
            j = i + 1 + (t - i * h);
            if (j >= S) j -= S;
        } else {
            i = t - S * h;
            j = i + S / 2;
        }
        sum += ld_dist<P>(base + i * L, base + j * L, L);
    }
    __shared__ int64_t part[LD_GROUP_THREADS / 32];
    for (int o = 16; o; o >>= 1) sum += __shfl_down_sync(FULL_MASK, sum, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t s = 0;
        for (int v = 0; v < LD_GROUP_THREADS / 32; ++v) s += part[v];
        sums[blockIdx.x] = s;
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------

static cudaError_t ld_pack(const LdGeom& g, const LdLevels& lv, uint32_t* dst, cudaStream_t s, int& n_launches) {
    if (lv.n == 0) return cudaSuccess;
    const int64_t threads = lv.n * g.W * 32;
    k_ld_pack<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(lv.p, lv.n, lv.stride, g.cells, g.W, g.P, dst);
    ++n_launches;
    return cudaGetLastError();
}

template <int P, bool FULL>
static cudaError_t ld_tile_launch(const LdTile& t, dim3 grid, size_t smem, cudaStream_t s) {
    cudaError_t e = cudaFuncSetAttribute(k_ld_tile<P, FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_ld_tile<P, FULL><<<grid, LD_THREADS, smem, s>>>(t);
    return cudaGetLastError();
}

template <bool FULL>
static cudaError_t ld_tile(const LdGeom& g, const LdTile& t, int64_t slices, cudaStream_t s, int& n_launches) {
    const dim3 grid((unsigned)((t.n_q + LD_QT - 1) / LD_QT), (unsigned)slices);
    const size_t smem = ld_tile_smem(g);
    ++n_launches;
    switch (g.P) {
        case 1: return ld_tile_launch<1, FULL>(t, grid, smem, s);
        case 2: return ld_tile_launch<2, FULL>(t, grid, smem, s);
        case 3: return ld_tile_launch<3, FULL>(t, grid, smem, s);
        default: return ld_tile_launch<4, FULL>(t, grid, smem, s);
    }
}

static LdTile ld_tile_args(const LdGeom& g, const LdLevels& a, const LdLevels& b, void* work) {
    LdTile t = {};
    t.qa = (const uint32_t*)work;
    t.ba = (const uint32_t*)((uint8_t*)work + align256(a.n * g.L * 4));
    t.n_q = a.n;
    t.n_b = b.n;
    t.L = g.L;
    t.pitch = ld_pitch(g);
    t.self_offset = -1;
    return t;
}

cudaError_t launch_level_distances(const LdGeom& g, const LdLevels& a, const LdLevels& b, int32_t* out, void* work,
                                   cudaStream_t s, int& n_launches) {
    LdTile t = ld_tile_args(g, a, b, work);
    cudaError_t e;
    if ((e = ld_pack(g, a, (uint32_t*)t.qa, s, n_launches)) != cudaSuccess) return e;
    if ((e = ld_pack(g, b, (uint32_t*)t.ba, s, n_launches)) != cudaSuccess) return e;
    t.slice_len = b.n;
    t.out = out;
    return ld_tile<true>(g, t, 1, s, n_launches);
}

cudaError_t launch_level_knn(const LdGeom& g, const LdLevels& q, const LdLevels& b, int k, int64_t self_offset,
                             int32_t* dist, int32_t* idx, void* work, cudaStream_t s, int& n_launches) {
    LdTile t = ld_tile_args(g, q, b, work);
    cudaError_t e;
    if ((e = ld_pack(g, q, (uint32_t*)t.qa, s, n_launches)) != cudaSuccess) return e;
    if ((e = ld_pack(g, b, (uint32_t*)t.ba, s, n_launches)) != cudaSuccess) return e;
    const LdSplit sp = ld_split(q.n, b.n);
    t.slice_len = sp.slice_len;
    t.k = k;
    t.self_offset = self_offset;
    t.out = dist;
    t.out_idx = idx;
    if (sp.slices > 1)
        t.partial = (uint64_t*)((uint8_t*)t.ba + align256(b.n * g.L * 4));
    if ((e = ld_tile<false>(g, t, sp.slices, s, n_launches)) != cudaSuccess || sp.slices == 1) return e;
    k_ld_merge<<<(unsigned)((q.n * 32 + 255) / 256), 256, 0, s>>>(t.partial, q.n, sp.slices, k, dist, idx);
    ++n_launches;
    return cudaGetLastError();
}

cudaError_t launch_level_groups(const LdGeom& g, const LdLevels& a, int64_t group_size, int64_t* sums, void* work,
                                cudaStream_t s, int& n_launches) {
    uint32_t* pk = (uint32_t*)work;
    cudaError_t e;
    if ((e = ld_pack(g, a, pk, s, n_launches)) != cudaSuccess) return e;
    const unsigned groups = (unsigned)(a.n / group_size);
    ++n_launches;
    switch (g.P) {
        case 1: k_ld_groups<1><<<groups, LD_GROUP_THREADS, 0, s>>>(pk, g.L, group_size, sums); break;
        case 2: k_ld_groups<2><<<groups, LD_GROUP_THREADS, 0, s>>>(pk, g.L, group_size, sums); break;
        case 3: k_ld_groups<3><<<groups, LD_GROUP_THREADS, 0, s>>>(pk, g.L, group_size, sums); break;
        default: k_ld_groups<4><<<groups, LD_GROUP_THREADS, 0, s>>>(pk, g.L, group_size, sums); break;
    }
    return cudaGetLastError();
}

}  // namespace pcgrl
