// Observation writer: Cropped + OneHotEncoding + ToImage (+ ControlWrapper target channels).
//
// Reference (relative to /root/reference/control_pcgrl/):
//   wrappers.py:407-437  Cropped._transform    out[o] = map[pos + o - obs//2] + 1, 0 when out of bounds
//   wrappers.py:232-257  OneHotEncoding        np.eye(dim)[.]  (dim = C+1 behind a crop, C otherwise)
//   wrappers.py:140-150  ToImage               channels last
//   control_wrappers.py:189-214 observe_metric_trgs   2*n_ctrl constant planes PREPENDED:
//                                              (trg / range, metric / range), tuple trg -> midpoint
// One thread per output pixel writes all of its channels (channels-last => contiguous per thread, and
// consecutive threads write consecutive pixels => coalesced stores).  The int8 grid rows are re-read
// through L1/L2; nothing else is loaded.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "pcgrl_device.cuh"

namespace pcgrl {

// An element of type T from a plane value or a small integer.  The 2-byte types (float16, bfloat16) round the FLOAT32
// element to nearest even, so a half observation is byte for byte the float32 one converted: x / range is rounded to
// float first.  (A double converted straight to a half type rounds once and differs on rare ties.)
template <typename T, typename S>
__device__ __forceinline__ T obs_elem(S x) {
    if constexpr (std::is_same_v<T, __half>) return __float2half_rn((float)x);
    else if constexpr (std::is_same_v<T, __nv_bfloat16>) return __float2bfloat16_rn((float)x);
    else return (T)x;
}
// the 16 bits of 1.0 in a 2-byte element type
template <typename T>
__host__ __device__ constexpr uint32_t half_one_bits() { return std::is_same_v<T, __half> ? 0x3C00u : 0x3F80u; }

struct ObsParams {
    int32_t ndim, d0, d1, d2, row_stride, n_tiles, n_stats;
    int32_t crop, o0, o1, o2;
    int32_t raw;                  // 1: write the tile code of each pixel (Cropped's output) instead of its one-hot record
    int32_t n_ctrl;
    int32_t ctrl_idx[PCGRL_MAX_STATS];
    double ctrl_range[PCGRL_MAX_STATS];
    int32_t targets_per_env;
    int64_t n_envs;
    const int8_t* grids;
    const int32_t* pos;
    const int32_t* stats;
    const double* targets;
    const uint8_t* static_mask;   // NULL: no static_builds plane
    const int32_t* holes;         // holey problems: [N,4] (3D: [N,6]) entrance / exit in bordered coordinates, else NULL
    int32_t border_tile;
    int32_t hole_ints;            // 4, or 6 for the 3D holey problems (foot tiles; the head is the tile above, z + 1)
    void* out;
};

// Observation of a list of envs (pcgrl_observe_envs): output row r shows env idx[r] of the shard.  A separate kernel
// argument after ObsParams / ObsVec, so that the identity instantiations (IDX == false, pcgrl_observe) keep their
// parameter offsets and code.  With IDX the writers' ObsParams::n_envs is the number of output rows.
struct ObsIdx {
    const int32_t* idx;   // [rows] env index of each output row
    int64_t n_envs;       // envs of the shard: nothing is loaded through an index outside [0, n_envs)
    int32_t* status;      // pcgrl_state.status or NULL: bit 64 for such an index
};
// the env that output row `row` shows, or -1 for an index outside the shard
template <bool IDX>
__device__ __forceinline__ int64_t obs_src(const ObsIdx& ix, int64_t row) {
    if constexpr (!IDX) {
        return row;
    } else {
        const int64_t e = ix.idx[row];
        return (uint64_t)e < (uint64_t)ix.n_envs ? e : -1;
    }
}
__device__ __forceinline__ void obs_flag_bad_index(const ObsIdx& ix) {
    if (ix.status) atomicOr(ix.status, 64);
}

template <typename T, bool IDX>
__global__ void __launch_bounds__(256) k_observe(const ObsParams p, const ObsIdx ix) {
    const int64_t pix_per_env = (int64_t)p.o0 * p.o1 * p.o2;
    const int64_t total = p.n_envs * pix_per_env;
    const int n_map_ch = p.raw ? 1 : (p.crop ? p.n_tiles + 1 : p.n_tiles);
    const int n_ch = 2 * p.n_ctrl + n_map_ch + (p.static_mask ? 1 : 0);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = i / pix_per_env;
        int r = (int)(i - row * pix_per_env);
        const int64_t env = obs_src<IDX>(ix, row);
        if (IDX && env < 0) {   // bad index: a zero record, nothing loaded
            if (r == 0) obs_flag_bad_index(ix);
            for (int c = 0; c < n_ch; ++c) ((T*)p.out)[i * n_ch + c] = obs_elem<T>(0);
            continue;
        }
        const int q2 = r % p.o2;
        r /= p.o2;
        const int q1 = r % p.o1;
        const int q0 = r / p.o1;
        int hot, frozen = 0;
        if (p.holes && p.ndim == 3) {
            // 3D holey problems: the bordered 3D map, entrance and exit dug two tiles high (foot + head,
            // HoleyRepresentation3D.dig_holes, envs/reps/wrappers.py:182-185), position shifted by the border
            const int32_t* h = p.holes + env * 6;
            int s0 = q0, s1 = q1, s2 = q2;
            if (p.crop) {
                const int32_t* pos = p.pos + env * 3;
                s0 = pos[0] + 1 + q0 - p.o0 / 2;
                s1 = pos[1] + 1 + q1 - p.o1 / 2;
                s2 = pos[2] + 1 + q2 - p.o2 / 2;
            }
            int v = -1;                                       // outside the bordered map: the crop's padding
            if ((unsigned)s0 < (unsigned)(p.d0 + 2) && (unsigned)s1 < (unsigned)(p.d1 + 2) &&
                (unsigned)s2 < (unsigned)(p.d2 + 2)) {
                if (s0 >= 1 && s0 <= p.d0 && s1 >= 1 && s1 <= p.d1 && s2 >= 1 && s2 <= p.d2) {
                    v = p.grids[env * p.row_stride + ((s0 - 1) * p.d1 + (s1 - 1)) * p.d2 + (s2 - 1)];
                } else {
                    const bool ent = (s0 == h[0] || s0 == h[0] + 1) && s1 == h[1] && s2 == h[2];
                    const bool ext = (s0 == h[3] || s0 == h[3] + 1) && s1 == h[4] && s2 == h[5];
                    v = (ent || ext) ? 0 : p.border_tile;
                }
            }
            hot = p.crop ? v + 1 : v;
        } else if (p.holes) {
            // holey problems (2D): the observed map is the bordered map with the two holes dug as empty tiles, and
            // the position is shifted by the border (HoleyRepresentation.get_observation, envs/reps/wrappers.py:153-160)
            const int32_t* h = p.holes + env * 4;
            int s0 = q0, s1 = q1;
            if (p.crop) {
                const int32_t* pos = p.pos + env * 3;
                s0 = pos[0] + 1 + q0 - p.o0 / 2;
                s1 = pos[1] + 1 + q1 - p.o1 / 2;
            }
            int v = -1;                                       // outside the bordered map: the crop's padding
            if ((unsigned)s0 < (unsigned)(p.d0 + 2) && (unsigned)s1 < (unsigned)(p.d1 + 2)) {
                if (s0 >= 1 && s0 <= p.d0 && s1 >= 1 && s1 <= p.d1)
                    v = p.grids[env * p.row_stride + (s0 - 1) * p.d1 + (s1 - 1)];
                else
                    v = ((s0 == h[0] && s1 == h[1]) || (s0 == h[2] && s1 == h[3])) ? 0 : p.border_tile;
            }
            hot = p.crop ? v + 1 : v;
        } else if (p.crop) {
            const int32_t* pos = p.pos + env * 3;
            const int s0 = pos[0] + q0 - p.o0 / 2, s1 = pos[1] + q1 - p.o1 / 2;
            const int s2 = (p.ndim == 3) ? pos[2] + q2 - p.o2 / 2 : 0;
            if ((unsigned)s0 < (unsigned)p.d0 && (unsigned)s1 < (unsigned)p.d1 && (unsigned)s2 < (unsigned)p.d2)
                hot = p.grids[env * p.row_stride + (s0 * p.d1 + s1) * p.d2 + s2] + 1;
            else
                hot = 0;
            if (p.static_mask) {
                // 'static_builds' (wrappers.py:451-459): the (dims+2) BORDERED mask goes through the same pad and
                // crop as the map, so window cell o shows bordered cell pos + o - obs//2 = map cell (that - 1);
                // border cells are always frozen (envs/reps/wrappers.py:310-312), beyond the border is padding (0)
                const int b0 = s0 - 1, b1 = s1 - 1, b2 = (p.ndim == 3) ? s2 - 1 : 0;
                const bool in_bordered = b0 >= -1 && b0 <= p.d0 && b1 >= -1 && b1 <= p.d1 &&
                                         (p.ndim != 3 || (b2 >= -1 && b2 <= p.d2));
                if (in_bordered) {
                    const bool inner = (unsigned)b0 < (unsigned)p.d0 && (unsigned)b1 < (unsigned)p.d1 &&
                                       (unsigned)b2 < (unsigned)p.d2;
                    frozen = inner ? p.static_mask[env * p.row_stride + (b0 * p.d1 + b1) * p.d2 + b2] != 0 : 1;
                }
            }
        } else {
            hot = p.grids[env * p.row_stride + (q0 * p.d1 + q1) * p.d2 + q2];
        }
        T* o = (T*)p.out + i * n_ch;
        for (int c = 0; c < p.n_ctrl; ++c) {
            const int k = p.ctrl_idx[c];
            const double* trg = p.targets + ((p.targets_per_env ? env * p.n_stats : 0) + k) * 2;
            double t = trg[0];
            if (!isnan(trg[1])) t = (trg[0] + trg[1]) / 2;
            o[2 * c] = obs_elem<T>(t / p.ctrl_range[c]);
            o[2 * c + 1] = obs_elem<T>((double)p.stats[env * p.n_stats + k] / p.ctrl_range[c]);
        }
        o += 2 * p.n_ctrl;
        if (p.raw) {
            o[0] = obs_elem<T>(hot);
        } else {
            for (int c = 0; c < n_map_ch; ++c) o[c] = obs_elem<T>(c == hot ? 1 : 0);
        }
        if (p.static_mask) o[n_map_ch] = obs_elem<T>(frozen);
    }
}

// ------------------------------------------------------------------------------------------------
// Staged writer (the one that normally runs).  The output is HBM-write bound (3 KB .. 17 KB per env against a
// 256-byte grid), so the stores must be full 128-bit coalesced vectors -- but a pixel's record (its channels) is
// 3 .. 9+ elements, never a vector.  Per trip a CTA therefore takes GB groups of G envs whose output is a whole
// number of 16-byte vectors, stages their grids / positions / ControlWrapper planes in shared memory, builds the
// records there (zero fill + one store per pixel, 32-bit index math with multiply-high divisions), and then
// streams the staged bytes to HBM with one 128-bit store per thread.  The one-thread-per-pixel kernel above,
// which stores element by element, stays as the fallback for unaligned output pointers / oversized groups.
// ------------------------------------------------------------------------------------------------
struct ObsVec {
    int32_t G, GB, E, pix, n_ch, n_map_ch, stage_bytes, planes_bytes;
    int32_t bits;                  // 1: two-tile crops from row bit masks + a 4-pixel record table (see k_observe_staged)
    int32_t lut_off;               // byte offset of that table in the dynamic shared memory
    uint32_t m_pix, m_o2, m_o12;   // floor(2^32 / d) of the divisors
};
__host__ __device__ inline uint32_t floor_magic(uint32_t d) { return d <= 1 ? 0xFFFFFFFFu : (uint32_t)(0x100000000ull / d); }
// n / d for any 32-bit n: the multiply-high by floor(2^32/d) is at most one too small
__device__ __forceinline__ uint32_t fdiv(uint32_t n, uint32_t d, uint32_t magic, uint32_t& rem) {
    uint32_t q = __umulhi(n, magic);
    rem = n - q * d;
    if (rem >= d) {
        ++q;
        rem -= d;
    }
    return q;
}
constexpr int OBS_MAX_CTA_ENVS = 64;   // GB * G
constexpr int OBS_THREADS = 256;

// IDX: rows come from ObsIdx (see there); only the staging loads below differ, the records and the copy-out are the
// same code over the trip's output rows
template <typename T, bool CROP, bool STATIC, bool D3, int ROWN /* 0, or 4 / 7 / 8 / 11 / 32: pixels per thread, all in one image row */,
          bool IDX>
__global__ void __launch_bounds__(OBS_THREADS) k_observe_staged(const ObsParams p, const ObsVec v, const ObsIdx ix) {
    extern __shared__ __align__(16) uint8_t obs_smem[];
    T* stage = (T*)obs_smem;                                         // [envs of the trip][pix][n_ch]
    T* s_planes = (T*)(obs_smem + v.stage_bytes);                    // [envs of the trip][2 * n_ctrl]
    // the trip's level grids (+ frozen-tile masks) and positions, staged with coalesced 128-bit loads so that the
    // per-pixel phase never waits on HBM
    const int8_t* s_grid = (const int8_t*)(obs_smem + v.stage_bytes + v.planes_bytes);
    const uint8_t* s_mask = (const uint8_t*)s_grid + (size_t)v.GB * v.G * p.row_stride;
    const int32_t* s_pos = (const int32_t*)(s_mask + (p.static_mask ? (size_t)v.GB * v.G * p.row_stride : 0));
    const int tid = threadIdx.x;
    const int envs_per_trip = v.GB * v.G;
    const int64_t trips = (p.n_envs + envs_per_trip - 1) / envs_per_trip;
    const int o12 = p.o1 * p.o2;
    const int n_pl = 2 * p.n_ctrl;
    // u8 one-hot records of 3 channels (binary behind a crop: the headline observation): 8 pixels are 24 bytes, built
    // in registers and stored as three 64-bit words -- no zero fill, no byte stores
    constexpr bool R8 = ROWN == 8 || ROWN == 32;
    const bool pack3 = sizeof(T) == 1 && R8 && !STATIC && v.n_ch == 3 && !p.raw && n_pl == 0;
    // uint8 tile codes (one byte per pixel): 8 pixels are one 64-bit word
    const bool pack1 = sizeof(T) == 1 && R8 && !STATIC && v.n_ch == 1 && p.raw && n_pl == 0;
    // 2-byte one-hot records of 3 channels on the row-mask path below: the u8 table's records, each byte widened
    const bool wide3 = sizeof(T) == 2 && ROWN == 8 && v.bits != 0 && !STATIC && v.n_ch == 3 && !p.raw && n_pl == 0;
    // Two-tile maps behind a crop (binary: the headline observation).  75 % of a 32x32 window on a 16x16 map is
    // padding, and the in-map / padding split of a warp's pixel groups made every warp run both record builders
    // (157 instructions per 24-byte group, issue-bound at 0.63 of the HBM peak).  Instead: the trip's map rows are
    // kept as 16-bit masks, a group's 8 tile bits and 8 inside bits are two clamped funnel shifts of its row, and
    // the records of 4 pixels at a time come from a 256-entry table indexed by (inside nibble, tile nibble) --
    // one instruction stream for padding and map pixels alike.
    const bool bits = v.bits != 0 && (pack3 || pack1 || wide3);
    uint16_t* s_rowbits = (uint16_t*)(obs_smem + v.lut_off + 256 * 16 + 256 * 4);   // [envs of the trip][d0]
    uint4* s_lut3 = (uint4*)(obs_smem + v.lut_off);                                  // 4 one-hot records (12 bytes)
    uint32_t* s_lut1 = (uint32_t*)(obs_smem + v.lut_off + 256 * 16);                 // 4 tile codes
    if (bits) {
        const uint32_t in4 = (uint32_t)tid >> 4, t4 = (uint32_t)tid & 15u;
        uint32_t rec[4], code = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t hot = ((in4 >> k) & 1u) ? 1u + ((t4 >> k) & 1u) : 0u;   // 0 = out of bounds, tile t -> t + 1
            rec[k] = 1u << (8 * hot);
            code |= hot << (8 * k);
        }
        s_lut3[tid] = make_uint4(rec[0] | (rec[1] << 24), (rec[1] >> 8) | (rec[2] << 16), (rec[2] >> 16) | (rec[3] << 8), 0u);
        s_lut1[tid] = code;
    }
    for (int64_t trip = blockIdx.x; trip < trips; trip += gridDim.x) {
        const int64_t env0 = trip * envs_per_trip;
        const int n_here = (int)min((int64_t)envs_per_trip, p.n_envs - env0);
        // the previous trip's bulk store has finished READING the stage (its global writes may still be in flight)
        if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncthreads();
        {
            const int nz = (pack3 || pack1 || wide3) ? 0 : (int)(((int64_t)n_here * v.E * (int64_t)sizeof(T) + 15) / 16);
            const uint4 z = make_uint4(0, 0, 0, 0);
            for (int i = tid; i < nz; i += OBS_THREADS) ((uint4*)stage)[i] = z;
            const int nv = n_here * (p.row_stride / 16);
            const uint4* g = (const uint4*)(p.grids + env0 * p.row_stride);
            if constexpr (IDX) {
                if (ix.status)
                    for (int i = tid; i < n_here; i += OBS_THREADS)
                        if (obs_src<IDX>(ix, env0 + i) < 0) obs_flag_bad_index(ix);
            }
            if (bits) {
                // one thread per map row: its tiles' low bits as a mask over x
                for (int i = tid; i < n_here * p.d0; i += OBS_THREADS) {
                    const int el = i / p.d0, y = i - el * p.d0;
                    const int64_t src = obs_src<IDX>(ix, env0 + el);
                    if (IDX && src < 0) {   // bad index: an empty map, nothing loaded
                        s_rowbits[i] = 0;
                        continue;
                    }
                    const int8_t* row = p.grids + src * p.row_stride + y * p.d1;
                    uint32_t m = 0;
                    if (p.d1 == 16) {
                        // one 128-bit load; the low bits of four tiles are gathered into a nibble by one multiply
                        // (bit 8j lands on 24 + j, the cross terms stay below bit 24)
                        const uint4 t = *(const uint4*)row;
                        const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
                        for (int k = 0; k < 4; ++k) m |= ((((w[k] & 0x01010101u) * 0x01020408u) >> 24) & 0xFu) << (4 * k);
                    } else {
#pragma unroll 4
                        for (int x = 0; x < p.d1; ++x) m |= (uint32_t)(row[x] & 1) << x;
                    }
                    s_rowbits[i] = (uint16_t)m;
                }
            } else if constexpr (IDX) {
                // one 128-bit copy per vector of each listed env's row (a bad index stages an empty map)
                const int vpr = p.row_stride / 16;
                for (int i = tid; i < nv; i += OBS_THREADS) {
                    const int el = i / vpr;
                    const int64_t src = obs_src<IDX>(ix, env0 + el);
                    ((uint4*)s_grid)[i] = src < 0 ? make_uint4(0, 0, 0, 0)
                                                  : ((const uint4*)p.grids)[src * vpr + (i - el * vpr)];
                }
            } else
            for (int i = tid; i < nv; i += OBS_THREADS) ((uint4*)s_grid)[i] = g[i];
            if (p.static_mask) {
                if constexpr (IDX) {
                    const int vpr = p.row_stride / 16;
                    for (int i = tid; i < nv; i += OBS_THREADS) {
                        const int el = i / vpr;
                        const int64_t src = obs_src<IDX>(ix, env0 + el);
                        ((uint4*)s_mask)[i] = src < 0 ? make_uint4(0, 0, 0, 0)
                                                      : ((const uint4*)p.static_mask)[src * vpr + (i - el * vpr)];
                    }
                } else {
                const uint4* m = (const uint4*)(p.static_mask + env0 * p.row_stride);
                for (int i = tid; i < nv; i += OBS_THREADS) ((uint4*)s_mask)[i] = m[i];
                }
            }
            if (p.crop) {
                if constexpr (IDX) {
                    for (int i = tid; i < n_here * 3; i += OBS_THREADS) {
                        const int el = i / 3;
                        const int64_t src = obs_src<IDX>(ix, env0 + el);
                        ((int32_t*)s_pos)[i] = src < 0 ? 0 : p.pos[src * 3 + (i - el * 3)];
                    }
                } else
                for (int i = tid; i < n_here * 3; i += OBS_THREADS) ((int32_t*)s_pos)[i] = p.pos[env0 * 3 + i];
            }
        }
        if (p.n_ctrl > 0) {
            for (int i = tid; i < n_here * p.n_ctrl; i += OBS_THREADS) {
                const int el = i / p.n_ctrl, c = i - el * p.n_ctrl;
                const int64_t env = obs_src<IDX>(ix, env0 + el);
                if (IDX && env < 0) {   // bad index: zero planes
                    s_planes[el * n_pl + 2 * c] = s_planes[el * n_pl + 2 * c + 1] = obs_elem<T>(0);
                    continue;
                }
                const int k = p.ctrl_idx[c];
                const double* trg = p.targets + ((p.targets_per_env ? env * p.n_stats : 0) + k) * 2;
                double t = trg[0];
                if (!isnan(trg[1])) t = (trg[0] + trg[1]) / 2;
                s_planes[el * n_pl + 2 * c] = obs_elem<T>(t / p.ctrl_range[c]);
                s_planes[el * n_pl + 2 * c + 1] = obs_elem<T>((double)p.stats[env * p.n_stats + k] / p.ctrl_range[c]);
            }
        }
        __syncthreads();
        // ---- records: the stage is zero-filled with 128-bit stores, then every pixel sets its ONE hot element ----
        // (a one-hot record is all zeros but one element, so building it is a single store at offset `hot`; the
        // ControlWrapper planes and the static_builds plane are the only other elements written.)  A thread takes
        // four consecutive pixels: the index math is paid once and the coordinates advance with carries.
        const int n_pix = n_here * v.pix;
        constexpr int PPT = ROWN ? ROWN : 4;   // pixels per thread
        for (int first = tid * PPT; first < n_pix; first += OBS_THREADS * PPT) {
            // coordinates of the first pixel: (env of the trip, q0, q1[, q2]); in 2D the image is (o0, o1).  (Hoisting
            // this out of the trips when the thread stride is a whole number of images costs 5 live registers and with
            // them a resident CTA: u8 binary-narrow 0.72 -> 0.66 of the HBM peak, f32 0.91 -> 0.86.)
            uint32_t r, q0, q1, q2 = 0;
            uint32_t el = fdiv((uint32_t)first, (uint32_t)v.pix, v.m_pix, r);
            if (D3) {
                uint32_t pr;
                q0 = fdiv(r, (uint32_t)o12, v.m_o12, pr);
                q1 = fdiv(pr, (uint32_t)p.o2, v.m_o2, q2);
            } else {
                q0 = fdiv(r, (uint32_t)p.o1, v.m_o12, q1);
            }
            const int8_t* grid = s_grid + el * p.row_stride;
            int c0 = 0, c1 = 0, c2 = 0;
            const int hb = p.holes ? 1 : 0;   // holey: positions are shifted by the border (wrappers.py:158-159)
            if (CROP) {
                c0 = s_pos[el * 3 + 0] + hb - p.o0 / 2;
                c1 = s_pos[el * 3 + 1] + hb - p.o1 / 2;
                if (D3) c2 = s_pos[el * 3 + 2] - p.o2 / 2;
            }
            T* o = stage + (size_t)first * v.n_ch + n_pl;
            if constexpr (ROWN != 0) {
                // the last image axis is a multiple of ROWN long: the pixels share a row, so the row test and the
                // row pointer are computed once and nothing carries
                bool row_ok = true;
                if (CROP) row_ok = D3 ? ((unsigned)(c0 + (int)q0) < (unsigned)p.d0 && (unsigned)(c1 + (int)q1) < (unsigned)p.d1)
                                      : (unsigned)(c0 + (int)q0) < (unsigned)p.d0;
                const int dl = D3 ? p.d2 : p.d1;
                const int sl = D3 ? c2 + (int)q2 : c1 + (int)q1;
                const int8_t* rowp = D3 ? grid + ((c0 + (int)q0) * p.d1 + (c1 + (int)q1)) * p.d2 : grid + (c0 + (int)q0) * p.d1;
                // which of the 8 pixels lie inside the map: most of a crop is padding (a 32x32 window on a 16x16 map
                // is 75 % out of bounds), and such pixels need no grid load -- a whole group outside is a constant
                const bool none_in = !row_ok || (CROP && (sl + 7 < 0 || sl >= dl));
                if (sizeof(T) == 1 && ROWN == 32 && bits) {
                    // A whole 32-pixel window row per thread (q1 == 0): the index math above is paid once per 32 pixels
                    // instead of once per 8 (the 1-byte tile codes ran at 6 instructions per output byte), the row's 32
                    // tile bits and 32 inside bits are two funnel shifts, eight table lookups give the records of four
                    // pixels each, and the row leaves as 128-bit stores.
                    const uint32_t rb = row_ok ? (uint32_t)s_rowbits[el * p.d0 + c0 + (int)q0] : 0u;
                    const uint32_t inr = row_ok ? ((1u << p.d1) - 1u) : 0u;
                    const uint32_t t32 = __funnelshift_rc(rb << 16, 0u, (uint32_t)(sl + 16));     // bit k = map column sl + k
                    const uint32_t in32 = __funnelshift_rc(inr << 16, 0u, (uint32_t)(sl + 16));
                    uint4* o16 = (uint4*)o;
                    if (pack3) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {      // 16 pixels = 48 bytes = three 128-bit stores
                            uint4 r[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int sh = 16 * h + 4 * j;
                                r[j] = s_lut3[(((in32 >> sh) & 0xFu) << 4) | ((t32 >> sh) & 0xFu)];
                            }
                            o16[3 * h + 0] = make_uint4(r[0].x, r[0].y, r[0].z, r[1].x);
                            o16[3 * h + 1] = make_uint4(r[1].y, r[1].z, r[2].x, r[2].y);
                            o16[3 * h + 2] = make_uint4(r[2].z, r[3].x, r[3].y, r[3].z);
                        }
                    } else {
                        uint32_t w[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            w[j] = s_lut1[(((in32 >> (4 * j)) & 0xFu) << 4) | ((t32 >> (4 * j)) & 0xFu)];
                        o16[0] = make_uint4(w[0], w[1], w[2], w[3]);
                        o16[1] = make_uint4(w[4], w[5], w[6], w[7]);
                    }
                } else if (ROWN == 8 && bits) {
                    // sl + 16 >= 0 (the window is at most 32 wide): bit k of the shifted row is map column sl + k
                    const uint32_t rb = row_ok ? (uint32_t)s_rowbits[el * p.d0 + c0 + (int)q0] : 0u;
                    const uint32_t inr = row_ok ? ((1u << p.d1) - 1u) : 0u;
                    const uint32_t t8 = __funnelshift_rc(rb << 16, 0u, (uint32_t)(sl + 16)) & 0xFFu;
                    const uint32_t in8 = __funnelshift_rc(inr << 16, 0u, (uint32_t)(sl + 16)) & 0xFFu;
                    const uint32_t ilo = ((in8 & 0xFu) << 4) | (t8 & 0xFu), ihi = (in8 & 0xF0u) | (t8 >> 4);
                    if constexpr (sizeof(T) == 2) {
                        // byte k of a table record (0 or 1) becomes 16-bit lane k: 0 or the bits of 1.0; 8 records
                        // are 48 bytes at a multiple of 48, three 128-bit stores
                        const uint4 a = s_lut3[ilo], b = s_lut3[ihi];
                        const uint32_t w[6] = {a.x, a.y, a.z, b.x, b.y, b.z};
                        uint32_t h[12];
#pragma unroll
                        for (int j = 0; j < 6; ++j) {
                            h[2 * j] = __byte_perm(w[j], 0u, 0x4140) * half_one_bits<T>();
                            h[2 * j + 1] = __byte_perm(w[j], 0u, 0x4342) * half_one_bits<T>();
                        }
                        uint4* o16 = (uint4*)o;
                        o16[0] = make_uint4(h[0], h[1], h[2], h[3]);
                        o16[1] = make_uint4(h[4], h[5], h[6], h[7]);
                        o16[2] = make_uint4(h[8], h[9], h[10], h[11]);
                    } else if (pack3) {
                        const uint4 a = s_lut3[ilo], b = s_lut3[ihi];
                        uint2* o8 = (uint2*)o;
                        o8[0] = make_uint2(a.x, a.y);
                        o8[1] = make_uint2(a.z, b.x);
                        o8[2] = make_uint2(b.y, b.z);
                    } else {
                        *(uint2*)o = make_uint2(s_lut1[ilo], s_lut1[ihi]);
                    }
                } else if (sizeof(T) == 1 && ROWN == 8 && pack3 && none_in) {
                    uint2* o8 = (uint2*)o;       // eight records "1 0 0"
                    o8[0] = make_uint2(0x01000001u, 0x00010000u);
                    o8[1] = make_uint2(0x00000100u, 0x01000001u);
                    o8[2] = make_uint2(0x00010000u, 0x00000100u);
                } else if (sizeof(T) == 1 && ROWN == 8 && pack1 && none_in) {
                    *(uint2*)o = make_uint2(0u, 0u);
                } else if (sizeof(T) == 1 && ROWN == 8 && pack3) {
                    // pixel k is the 24-bit value 1 << (8 * hot_k); four of them make three 32-bit words
                    uint32_t px[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const bool inside = row_ok && (!CROP || (unsigned)(sl + k) < (unsigned)dl);
                        const int hot = inside ? rowp[sl + k] + (CROP ? 1 : 0) : 0;
                        px[k] = 1u << (8 * hot);
                    }
                    uint32_t w[6];
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        w[3 * h + 0] = px[4 * h] | (px[4 * h + 1] << 24);
                        w[3 * h + 1] = (px[4 * h + 1] >> 8) | (px[4 * h + 2] << 16);
                        w[3 * h + 2] = (px[4 * h + 2] >> 16) | (px[4 * h + 3] << 8);
                    }
                    uint2* o8 = (uint2*)o;       // byte offset first * 3 with first % 8 == 0: 8-byte aligned
                    o8[0] = make_uint2(w[0], w[1]);
                    o8[1] = make_uint2(w[2], w[3]);
                    o8[2] = make_uint2(w[4], w[5]);
                } else if (sizeof(T) == 1 && ROWN == 8 && pack1) {
                    uint32_t lo = 0, hi = 0;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const bool inside = row_ok && (!CROP || (unsigned)(sl + k) < (unsigned)dl);
                        const uint32_t hot = inside ? (uint32_t)(rowp[sl + k] + (CROP ? 1 : 0)) : 0u;
                        if (k < 4) lo |= hot << (8 * k);
                        else hi |= hot << (8 * (k - 4));
                    }
                    *(uint2*)o = make_uint2(lo, hi);
                } else
#pragma unroll
                for (int k = 0; k < ROWN; ++k) {
                    const bool inside = row_ok && (!CROP || (unsigned)(sl + k) < (unsigned)dl);
                    const int hot = inside ? rowp[sl + k] + (CROP ? 1 : 0) : 0;
                    for (int c = 0; c < n_pl; ++c) o[k * v.n_ch - n_pl + c] = s_planes[el * n_pl + c];
                    if constexpr (sizeof(T) == 2) o[k * v.n_ch + hot] = obs_elem<T>(1);   // no 2-byte tile codes
                    else o[k * v.n_ch + (p.raw ? 0 : hot)] = p.raw ? obs_elem<T>(hot) : obs_elem<T>(1);
                    if (STATIC) {   // see k_observe: the bordered frozen-tile mask through the same crop
                        const int s0 = c0 + (int)q0, s1 = D3 ? c1 + (int)q1 : sl + k, s2 = D3 ? sl + k : 0;
                        const int b0 = s0 - 1, b1 = s1 - 1, b2 = D3 ? s2 - 1 : 0;
                        const bool in_bordered = b0 >= -1 && b0 <= p.d0 && b1 >= -1 && b1 <= p.d1 &&
                                                 (!D3 || (b2 >= -1 && b2 <= p.d2));
                        if (in_bordered) {
                            const bool inner = (unsigned)b0 < (unsigned)p.d0 && (unsigned)b1 < (unsigned)p.d1 &&
                                               (unsigned)b2 < (unsigned)p.d2;
                            if (!inner || s_mask[el * p.row_stride + (b0 * p.d1 + b1) * p.d2 + b2] != 0)
                                o[k * v.n_ch + v.n_map_ch] = obs_elem<T>(1);
                        }
                    }
                }
            } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (first + k < n_pix) {
                    const int s0 = c0 + (int)q0, s1 = c1 + (int)q1, s2 = D3 ? c2 + (int)q2 : 0;
                    bool inside = true;
                    if (CROP)
                        inside = (unsigned)s0 < (unsigned)p.d0 && (unsigned)s1 < (unsigned)p.d1 &&
                                 (!D3 || (unsigned)s2 < (unsigned)p.d2);
                    const int cell = D3 ? (s0 * p.d1 + s1) * p.d2 + s2 : s0 * p.d1 + s1;
                    // crop: channel 0 = out of bounds, tile t -> channel t + 1 (wrappers.py:420-437); else channel = tile
                    int hot;
                    if (p.holes) {
                        // holey (2D): (s0, s1) address the BORDERED map -- level inside, border tile around it, the
                        // two holes empty (see k_observe)
                        const int64_t src = obs_src<IDX>(ix, env0 + el);
                        const int32_t* h = p.holes + src * 4;
                        int val = -1;
                        if ((unsigned)s0 < (unsigned)(p.d0 + 2) && (unsigned)s1 < (unsigned)(p.d1 + 2)) {
                            if (s0 >= 1 && s0 <= p.d0 && s1 >= 1 && s1 <= p.d1)
                                val = grid[(s0 - 1) * p.d1 + (s1 - 1)];
                            else   // (a bad index: no holes)
                                val = ((!IDX || src >= 0) &&
                                       ((s0 == h[0] && s1 == h[1]) || (s0 == h[2] && s1 == h[3]))) ? 0 : p.border_tile;
                        }
                        hot = CROP ? val + 1 : val;
                    } else {
                        hot = inside ? grid[cell] + (CROP ? 1 : 0) : 0;
                    }
                    for (int c = 0; c < n_pl; ++c) o[k * v.n_ch - n_pl + c] = s_planes[el * n_pl + c];
                    if constexpr (sizeof(T) == 2) o[k * v.n_ch + hot] = obs_elem<T>(1);   // no 2-byte tile codes
                    else o[k * v.n_ch + (p.raw ? 0 : hot)] = p.raw ? obs_elem<T>(hot) : obs_elem<T>(1);
                    if (STATIC) {   // see k_observe: the bordered frozen-tile mask through the same crop
                        const int b0 = s0 - 1, b1 = s1 - 1, b2 = D3 ? s2 - 1 : 0;
                        const bool in_bordered = b0 >= -1 && b0 <= p.d0 && b1 >= -1 && b1 <= p.d1 &&
                                                 (!D3 || (b2 >= -1 && b2 <= p.d2));
                        if (in_bordered) {
                            const bool inner = (unsigned)b0 < (unsigned)p.d0 && (unsigned)b1 < (unsigned)p.d1 &&
                                               (unsigned)b2 < (unsigned)p.d2;
                            if (!inner || s_mask[el * p.row_stride + (b0 * p.d1 + b1) * p.d2 + b2] != 0)
                                o[k * v.n_ch + v.n_map_ch] = obs_elem<T>(1);
                        }
                    }
                    // next pixel: the last image axis is fastest
                    bool wrap_env = false;
                    if (D3) {
                        if (++q2 == (uint32_t)p.o2) {
                            q2 = 0;
                            if (++q1 == (uint32_t)p.o1) {
                                q1 = 0;
                                wrap_env = ++q0 == (uint32_t)p.o0;
                            }
                        }
                    } else if (++q1 == (uint32_t)p.o1) {
                        q1 = 0;
                        wrap_env = ++q0 == (uint32_t)p.o0;
                    }
                    if (wrap_env) {   // the quad continues in the next env of the trip
                        q0 = 0;
                        ++el;
                        grid += p.row_stride;
                        if (CROP && first + k + 1 < n_pix) {
                            c0 = s_pos[el * 3 + 0] + hb - p.o0 / 2;
                            c1 = s_pos[el * 3 + 1] + hb - p.o1 / 2;
                            if (D3) c2 = s_pos[el * 3 + 2] - p.o2 / 2;
                        }
                    }
                }
            }
            }
        }
        // ---- copy-out: ONE bulk asynchronous copy of the whole stage (cp.async.bulk shared -> global, the TMA engine;
        // SASS UBLKCP), issued by one thread, so no thread spends issue slots on the 128-bit load / store pairs and
        // the next trip's staging overlaps the drain.  Generic-proxy writes to shared memory must be fenced for the
        // async proxy before the barrier.
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        const int64_t elems = (int64_t)n_here * v.E;
        const int n_vec = (int)(elems * (int64_t)sizeof(T) / 16);
        uint4* dst = (uint4*)((T*)p.out + env0 * v.E);
        if (tid == 0 && n_vec > 0) {
            const uint32_t src_s = (uint32_t)__cvta_generic_to_shared(stage);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         :: "l"(dst), "r"(src_s), "r"(n_vec * 16) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        // a partly filled last group may end inside a vector: element-wise tail
        const int done = n_vec * (16 / (int)sizeof(T));
        for (int i = done + tid; i < (int)elems; i += OBS_THREADS) ((T*)p.out + env0 * v.E)[i] = stage[i];
    }
    if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the stage must outlive its last reader
}

template <typename T, bool IDX>
static cudaError_t launch_vec(const ObsParams& p, const ObsIdx& ix, cudaStream_t s, bool& done) {
    done = false;
    if ((uintptr_t)p.out % 16) return cudaSuccess;
    const int64_t pix = (int64_t)p.o0 * p.o1 * p.o2;
    const int n_map_ch = p.raw ? 1 : (p.crop ? p.n_tiles + 1 : p.n_tiles);
    const int n_ch = 2 * p.n_ctrl + n_map_ch + (p.static_mask ? 1 : 0);
    const int64_t E = pix * n_ch;
    ObsVec v;
    v.G = 1;
    while ((v.G * E * (int64_t)sizeof(T)) % 16) v.G *= 2;          // <= 16
    const int64_t group_bytes = v.G * E * (int64_t)sizeof(T);
    if (group_bytes > 160 * 1024) return cudaSuccess;               // oversized: the scalar kernel handles it
    v.GB = 1;
    while (v.GB * v.G * 2 <= OBS_MAX_CTA_ENVS && (v.GB * 2) * group_bytes <= 24 * 1024) v.GB *= 2;
    v.E = (int)E;
    v.pix = (int)pix;
    v.n_ch = n_ch;
    v.n_map_ch = n_map_ch;
    v.stage_bytes = (int)(v.GB * group_bytes);
    v.m_pix = floor_magic((uint32_t)pix);
    v.m_o2 = floor_magic((uint32_t)p.o2);
    v.m_o12 = floor_magic((uint32_t)(p.o1 * p.o2));   // 2D: o2 == 1, i.e. the magic of o1
    v.planes_bytes = (v.GB * v.G * 2 * p.n_ctrl * (int)sizeof(T) + 15) / 16 * 16;
    int dyn = v.stage_bytes + v.planes_bytes + v.GB * v.G * (p.row_stride * (p.static_mask ? 2 : 1) + 12);
    // two-tile crops of maps up to 16 wide in windows up to 32 wide (u8 / 2-byte one-hot or u8 codes, no extra planes):
    // row-mask path
    v.bits = sizeof(T) <= 2 && p.crop && p.ndim == 2 && p.n_tiles == 2 && p.d1 <= 16 && p.o1 <= 32 && p.o1 % 8 == 0 &&
             !p.static_mask && !p.holes && p.n_ctrl == 0 && (p.raw ? n_ch == 1 : n_ch == 3);
    v.lut_off = (dyn + 15) / 16 * 16;
    if (v.bits) dyn = v.lut_off + 256 * 16 + 256 * 4 + (v.GB * v.G * p.d0 * 2 + 15) / 16 * 16;
    const bool d3 = p.ndim == 3, st = p.static_mask != nullptr, cr = p.crop != 0;
    const int last_axis = d3 ? p.o2 : p.o1;
    // 8 pixels per thread only for 1-byte elements: with 4-byte elements a thread's 8 records are 8 * n_ch words
    // apart and the shared-memory stores conflict (f32 binary-narrow 4.05e8 -> 3.68e8 obs/s with 8, u8 8.8e8 -> 9.7e8)
    const int rown = p.holes ? 0   // the border frame is only handled by the general path
                   : (sizeof(T) == 1 && last_axis % 8 == 0) ? 8 : (last_axis % 4 == 0 ? 4 : 0);
#define OBS_PICK(RN)                                                                                                     \
    (cr ? (st ? (d3 ? k_observe_staged<T, true, true, true, RN, IDX> : k_observe_staged<T, true, true, false, RN, IDX>)  \
              : (d3 ? k_observe_staged<T, true, false, true, RN, IDX> : k_observe_staged<T, true, false, false, RN, IDX>)) \
        : (d3 ? k_observe_staged<T, false, false, true, RN, IDX> : k_observe_staged<T, false, false, false, RN, IDX>))
    void (*kern)(const ObsParams, const ObsVec, const ObsIdx);
    if constexpr (sizeof(T) == 2) {
        // float16 / bfloat16: only the kernels this choice reaches are instantiated.  B200 at 1000 W, 262 144 envs,
        // bf16 (profiles/r03_observe_half_ab.txt):
        // - two-tile crops take the row-mask path, 8 pixels (48 bytes, three 128-bit stores) per thread: binary-narrow
        //   32x32 0.2764 / 0.2759 ms against 0.3231 / 0.3230 ms on the 4-pixel path;
        // - 14-wide 3D windows take 7 pixels per thread: minecraft 14^3 1.0209 / 1.0181 ms against 1.8901 / 1.8919 ms;
        // - 4 pixels per thread otherwise (24 bytes of 3-channel records, the bank pattern of the u8 path's 8):
        //   binary-wide + 2 controls 0.2696 / 0.2693 ms against 0.4347 / 0.4341 ms with 8;
        // - 22-wide windows keep the general path: zelda 22x22 0.4704 / 0.4707 ms against 0.4919 / 0.4916 ms with 11.
        if (v.bits) kern = k_observe_staged<T, true, false, false, 8, IDX>;
        else if (!p.holes && !st && cr && d3 && p.o2 == 14) kern = k_observe_staged<T, true, false, true, 7, IDX>;
        else kern = rown == 4 ? OBS_PICK(4) : OBS_PICK(0);
    } else {
        kern = rown == 8 ? OBS_PICK(8) : (rown == 4 ? OBS_PICK(4) : OBS_PICK(0));
    }
#undef OBS_PICK
    if constexpr (sizeof(T) == 1) {
        // u8 windows 22 wide (zelda 7x11 behind its 22x22 crop: neither a multiple of 8 nor of 4, so it ran the 4-pixel
        // path with carries): half a window row (11 pixels) per thread, 0.2339 ms against 0.3465 ms with 4 and 0.2607 ms
        // with a whole row (profiles/r02_observe_row22.txt)
        if (rown == 0 && p.o1 == 22 && !d3 && !st && cr && !p.holes) kern = k_observe_staged<T, true, false, false, 11, IDX>;
        // ... and the 3D maze's 14-wide last axis (14^3 window of a 14^3 level): 7 pixels per thread, 0.776 ms against
        // 1.6133 ms with 4 and 0.8206 ms with 14 (profiles/r02_observe_row14.txt)
        if (rown == 0 && d3 && p.o2 == 14 && !st && cr && !p.holes) kern = k_observe_staged<T, true, false, true, 7, IDX>;
        // row-mask crops whose window is exactly 32 wide (binary 16x16 behind its 32x32 crop): a whole window row per
        // thread, 0.1649 ms against 0.1852 ms with 8 pixels per thread (profiles/r02_observe_row32.jsonl)
        if (v.bits && rown == 8 && p.o1 == 32 && !d3 && !st && cr) kern = k_observe_staged<T, true, false, false, 32, IDX>;
    }
    cudaError_t e;
    if (dyn > 48 * 1024 &&
        (e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn)) != cudaSuccess)
        return e;
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, OBS_THREADS, dyn)) != cudaSuccess) return e;
    if (per_sm < 1) return cudaSuccess;
    int n_sm = 0;
    if ((e = sm_count(n_sm)) != cudaSuccess) return e;
    const int64_t trips = (p.n_envs + v.GB * v.G - 1) / (v.GB * v.G);
    const int64_t cap = (int64_t)n_sm * per_sm;
    const unsigned blocks = (unsigned)(trips < cap ? trips : cap);
    kern<<<blocks, OBS_THREADS, dyn, s>>>(p, v, ix);
    done = true;
    return cudaGetLastError();
}

template <bool IDX>
static cudaError_t launch_writers(const ObsParams& p, const ObsIdx& ix, int out_kind, bool holey3d, int64_t total,
                                  cudaStream_t s) {
    // the staged writer knows the 2D border frame only; the bordered 3D map goes through the pixel-per-thread kernel
    if (!holey3d) {
        bool done = false;
        cudaError_t e = (out_kind == 0 || out_kind == 3) ? launch_vec<uint8_t, IDX>(p, ix, s, done)
                      : out_kind == 1 ? launch_vec<float, IDX>(p, ix, s, done)
                      : out_kind == 2 ? launch_vec<double, IDX>(p, ix, s, done)
                      : out_kind == 5 ? launch_vec<__half, IDX>(p, ix, s, done)
                      : out_kind == 6 ? launch_vec<__nv_bfloat16, IDX>(p, ix, s, done) : cudaErrorInvalidValue;
        if (e != cudaSuccess || done) return e;
    }
    const int64_t want = (total + 255) / 256;
    const unsigned blocks = (unsigned)(want < 148 * 32 ? want : 148 * 32);
    if (out_kind == 0 || out_kind == 3)
        k_observe<uint8_t, IDX><<<blocks, 256, 0, s>>>(p, ix);
    else if (out_kind == 1)
        k_observe<float, IDX><<<blocks, 256, 0, s>>>(p, ix);
    else if (out_kind == 2)
        k_observe<double, IDX><<<blocks, 256, 0, s>>>(p, ix);
    else if (out_kind == 5)
        k_observe<__half, IDX><<<blocks, 256, 0, s>>>(p, ix);
    else if (out_kind == 6)
        k_observe<__nv_bfloat16, IDX><<<blocks, 256, 0, s>>>(p, ix);
    else
        return cudaErrorInvalidValue;
    return cudaGetLastError();
}

// What launch_observe refuses (it then returns cudaErrorInvalidValue), as a message; NULL if it launches.  Host only,
// so that pcgrl_lookahead_obs can check the observation before its first launch.
const char* obs_args_error(const pcgrl_config& cfg, const pcgrl_state& st, const pcgrl_obs_args& a) {
    const bool holey3d = cfg.problem == PCGRL_PROB_MINECRAFT_3D_HOLEY_MAZE || cfg.problem == PCGRL_PROB_MINECRAFT_3D_DUNGEON_HOLEY;
    const bool holey = cfg.problem == PCGRL_PROB_BINARY_HOLEY || holey3d;
    if (holey) {
        if (!st.holes || cfg.ndim != (holey3d ? 3 : 2) || a.static_channel)
            return "a holey problem's observation needs holes and has no static_builds plane";
        if (a.holey_border_tile < 0 || a.holey_border_tile >= cfg.n_tiles) return "holey_border_tile out of range";
    }
    if (a.static_channel && (!a.crop || !st.static_mask)) return "the static_builds plane needs a crop and a static mask";
    const int grow = holey ? 2 : 0;   // without a crop the whole (bordered) map is observed
    const int o2 = cfg.ndim == 3 ? a.obs_dims[2] : 1, d2 = cfg.ndim == 3 ? cfg.dims[2] : 1;
    if (!a.crop && (a.obs_dims[0] != cfg.dims[0] + grow || a.obs_dims[1] != cfg.dims[1] + grow ||
                    o2 != d2 + (holey3d ? grow : 0)))
        return "without a crop obs_dims must be the (bordered) map dims";
    if ((a.out_kind == 0 || a.out_kind == 3) && a.n_ctrl > 0) return "uint8 observations have no target planes";
    return nullptr;   // an out_kind outside 0..3, 5, 6 fails at the launch (and passes when there is nothing to write)
}

// env_idx: NULL observes every env of the shard into row env; else n_idx rows, row j showing env env_idx[j]
cudaError_t launch_observe(const pcgrl_config& cfg, const pcgrl_state& st, const pcgrl_obs_args& a, cudaStream_t s,
                           const int32_t* env_idx, int64_t n_idx) {
    if (obs_args_error(cfg, st, a)) return cudaErrorInvalidValue;
    ObsParams p;
    p.ndim = cfg.ndim;
    p.d0 = cfg.dims[0];
    p.d1 = cfg.dims[1];
    p.d2 = cfg.ndim == 3 ? cfg.dims[2] : 1;
    p.row_stride = cfg.row_stride;
    p.n_tiles = cfg.n_tiles;
    p.n_stats = cfg.n_stats;
    p.crop = a.crop;
    p.raw = a.out_kind == 3;
    p.o0 = a.obs_dims[0];
    p.o1 = a.obs_dims[1];
    p.o2 = cfg.ndim == 3 ? a.obs_dims[2] : 1;
    p.n_ctrl = a.n_ctrl;
    for (int i = 0; i < PCGRL_MAX_STATS; ++i) {
        p.ctrl_idx[i] = a.ctrl_idx[i];
        p.ctrl_range[i] = a.ctrl_range[i];
    }
    p.targets_per_env = cfg.targets_per_env;
    p.n_envs = env_idx ? n_idx : st.n_envs;   // output rows
    p.grids = st.grids;
    p.pos = st.pos;
    p.stats = st.stats;
    p.targets = st.targets;
    p.holes = nullptr;
    p.border_tile = 0;
    p.hole_ints = 4;
    const bool holey3d = cfg.problem == PCGRL_PROB_MINECRAFT_3D_HOLEY_MAZE || cfg.problem == PCGRL_PROB_MINECRAFT_3D_DUNGEON_HOLEY;
    const bool holey = cfg.problem == PCGRL_PROB_BINARY_HOLEY || holey3d;
    if (holey) {
        p.hole_ints = holey3d ? 6 : 4;
        p.holes = st.holes;
        p.border_tile = a.holey_border_tile;
    }
    p.static_mask = a.static_channel ? st.static_mask : nullptr;
    p.out = a.out;
    const int64_t total = p.n_envs * (int64_t)p.o0 * p.o1 * p.o2;
    if (total == 0) return cudaSuccess;
    return env_idx ? launch_writers<true>(p, ObsIdx{env_idx, st.n_envs, st.status}, a.out_kind, holey3d, total, s)
                   : launch_writers<false>(p, ObsIdx{nullptr, st.n_envs, nullptr}, a.out_kind, holey3d, total, s);
}

}  // namespace pcgrl
