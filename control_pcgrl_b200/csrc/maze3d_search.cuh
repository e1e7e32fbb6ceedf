// minecraft_3D_maze search machinery (bit-mask level, FIFO label-correcting player search, far tile), shared by the
// plain problem (step_maze3d.cu) and the holey problems on the bordered map (step_maze3d_holey.cu).
#pragma once
#include "step_search.cuh"

namespace pcgrl {

constexpr int MAZE_QCAP = 256;    // FIFO ring capacity (entries); measured maximum with push filtering: 50
// small CTAs, several per SM: finer-grained tile barriers.  A/B on B200 (14^3, 65 536 envs): 4 / 6 / 8 / 16 warps per
// CTA -> 1.81 / 2.13 / 2.05 / 1.41e7 env-steps/s
constexpr int MAZE_WARPS = 6;
constexpr int MAZE_CTAS_PER_SM = 32 / MAZE_WARPS;
constexpr int MAZE_MAX_CTAS = 160 * MAZE_CTAS_PER_SM;   // sizes the global scratch (>= 148 SMs x 8 CTAs)
constexpr int MAZE_NJ_SLICE = 16 * 16 * 16 * 2;         // bytes of nj per warp (maps up to 16^3)
constexpr int MAZE_ORDER_SLICE = (16 / 2 + 1) * 16 * 16 * 2;   // bytes of the first-recording order list per warp
constexpr int MAZE_PAR_SLICE = 16 * 16 * 16 * 2;        // bytes of the parent pointers per warp (holey maze only)
constexpr int MAZE_SLICE = MAZE_NJ_SLICE + MAZE_ORDER_SLICE + MAZE_PAR_SLICE;

struct MazeLayout {
    int best, q_cl, nj, order, q_nj, q_par, col, row, total, order_cap, best_bytes;
};
__host__ __device__ inline MazeLayout maze_layout(int Z, int Y, int X, int row_stride) {
    MazeLayout L;
    const int cells = Z * Y * X;
    int bb = 2 * cells;
    if (bb < row_stride) bb = row_stride;      // the raw grid is staged here first
    if (bb < Z * Y * 32) bb = Z * Y * 32;      // ... and the region count's 32-bit run parents live here last
    bb = (bb + 15) / 16 * 16;
    L.best_bytes = bb;
    L.order_cap = (Z / 2 + 1) * Y * X;
    int o = 0;
    L.best = o;  o += bb;
    L.q_cl = o;  o += 4 * MAZE_QCAP;
    L.nj = -1;   // global scratch, see make_ctx
    L.order = -1;   // global scratch too: appended by lane 0, re-read a handful of times per grid
    L.q_nj = o;  o += 2 * MAZE_QCAP;
    L.q_par = o; o += 2 * MAZE_QCAP;   // parent cell of each queued entry (only filled by search<true>)
    L.col = o;   o += 2 * Y * X;
    L.row = o;   o += 2 * Z * Y;
    L.total = (o + 15) / 16 * 16;
    return L;
}

struct Maze3DProb {
    static constexpr int K = 3;   // regions, path-length, n_jump

    struct Ctx {
        int Z, Y, X, cells, R;
        uint32_t magic_xy, magic_x;
        uint16_t *best, *nj, *order, *par, *q_nj, *q_par, *col, *row;
        uint32_t* q_cl;
        int best_bytes, order_cap;
        int32_t* status;
    };

    __device__ static Ctx make_ctx(const KParams& p, uint8_t* ws, int global_warp) {
        return make_ctx_dims(p, ws, global_warp, p.d0, p.d1, p.d2);
    }
    // (Z, Y, X): the dimensions the search runs on -- the map's own, or the bordered map's for the holey problems
    __device__ static Ctx make_ctx_dims(const KParams& p, uint8_t* ws, int global_warp, int Z, int Y, int X) {
        Ctx c;
        c.Z = Z; c.Y = Y; c.X = X;
        c.cells = Z * Y * X;
        c.R = c.Z * c.Y;
        c.magic_xy = div_magic(c.X * c.Y);
        c.magic_x = div_magic(c.X);
        const MazeLayout L = maze_layout(c.Z, c.Y, c.X, p.row_stride);
        c.best = (uint16_t*)(ws + L.best);
        c.q_cl = (uint32_t*)(ws + L.q_cl);
        c.nj = (uint16_t*)((uint8_t*)p.scratch + (size_t)global_warp * MAZE_SLICE);
        c.order = (uint16_t*)((uint8_t*)p.scratch + (size_t)global_warp * MAZE_SLICE + MAZE_NJ_SLICE);
        c.par = (uint16_t*)((uint8_t*)p.scratch + (size_t)global_warp * MAZE_SLICE + MAZE_NJ_SLICE + MAZE_ORDER_SLICE);
        c.q_nj = (uint16_t*)(ws + L.q_nj);
        c.q_par = (uint16_t*)(ws + L.q_par);
        c.col = (uint16_t*)(ws + L.col);
        c.row = (uint16_t*)(ws + L.row);
        c.best_bytes = L.best_bytes;
        c.order_cap = L.order_cap;
        c.status = p.status;
        return c;
    }

    // ---- helper_3D._passable for one direction: foothold reached from (x, y, z) going (dx, dy) ----------
    // Returns false if the direction offers no move; else the foothold cell index, the number of path
    // entries the move appends (1 walk, 2 stairs / level jump, 3 jump up / down) and whether it is a jump.
    // Branch-free: with w = the neighbour column's AIR bits z-2 .. z+3 (bits below 0 and from Z up read as "not
    // AIR", which is what the reference's explicit range tests amount to) the four kinds of move are mutually
    // exclusive bit patterns --
    //   walk       !w1  w2  w3                      (:229-237)      step down  !w0  w1  w2  w3   (:243-252)
    //   step up    !w2  w3  w4  and head-room c0[z+2] (:259-266)    jump        w0..w4 all AIR, c0[z+2], landing column in range (:279-288)
    // and so are the three landings of a jump on the column two cells away (u = its bits z-2 .. z+3):
    //   level !u1 u2 u3 u4 (:289-296)   up !u2 u3 u4 u5 (:297-304)   down !u0 u1 u2 u3 (:305-312)
    // so the four lanes of a pop run one straight instruction stream instead of a cascade of divergent tests.
    __device__ static __forceinline__ bool move(const Ctx& c, int x, int y, int z, int dx, int dy, int& ncell,
                                                int& cost, int& jump) {
        const int nx = x + dx, ny = y + dy;
        if (nx < 0 || ny < 0 || nx >= c.X || ny >= c.Y) return false;                    // :225
        const uint32_t cn = c.col[ny * c.X + nx], c0 = c.col[y * c.X + x];
        const uint32_t w = ((cn << 2) >> z) & 0x3Fu;
        const uint32_t h2 = (c0 >> (z + 2)) & 1u;
        const uint32_t w0 = w & 1u, w1 = (w >> 1) & 1u, w2 = (w >> 2) & 1u, w3 = (w >> 3) & 1u, w4 = (w >> 4) & 1u;
        const uint32_t walk = (w1 ^ 1u) & w2 & w3;
        const uint32_t down = (w0 ^ 1u) & w1 & w2 & w3;
        const uint32_t up = (w2 ^ 1u) & w3 & w4 & h2;
        const int jx = nx + dx, jy = ny + dy;
        const bool j_in = jx >= 0 && jy >= 0 && jx < c.X && jy < c.Y;
        const uint32_t jp = ((w & 0x1Fu) == 0x1Fu) & h2 & (uint32_t)j_in;
        const uint32_t cj = j_in ? c.col[jy * c.X + jx] : 0u;
        const uint32_t u = ((cj << 2) >> z) & 0x3Fu;
        const uint32_t u0 = u & 1u, u1 = (u >> 1) & 1u, u2 = (u >> 2) & 1u, u3 = (u >> 3) & 1u, u4 = (u >> 4) & 1u,
                       u5 = (u >> 5) & 1u;
        const uint32_t j_level = jp & (u1 ^ 1u) & u2 & u3 & u4;
        const uint32_t j_up = jp & (u2 ^ 1u) & u3 & u4 & u5;
        const uint32_t j_down = jp & (u0 ^ 1u) & u1 & u2 & u3;
        const uint32_t landed = j_level | j_up | j_down;
        jump = (int)jp;
        const int nz = z + (int)(up | j_up) - (int)(down | j_down);
        cost = (int)(walk + 2u * (down | up | j_level) + 3u * (j_up | j_down));
        ncell = landed ? (nz * c.Y + jy) * c.X + jx : (nz * c.Y + ny) * c.X + nx;
        return (walk | down | up | landed) != 0u;
    }

    // ---- helper_3D.run_dijkstra from `start` (warp-uniform FIFO; lanes 0..3 evaluate the 4 directions) -----
    // Leaves order[0..n) = cells in first-recording order, best[c] & 0x7FFF = len(paths[c]), nj[c] = jumps[c].
    // PARENTS: also leave par[c] = the cell the recorded path reaches c from (par[start] = start).  The start tile
    // needs head-room like every recorded tile (helper_3D.py:443-445), else nothing is recorded.
    // One pop per round: the queue rarely holds more than 1-3 entries, and popping up to 32 per round measured
    // 1.45e7 against 2.25e7 env-steps/s on B200 (14^3, 65 536 envs).
    template <bool PARENTS = false>
    __device__ static int search(Ctx& c, int start, int lane, bool& overflow) {
        const int XY = c.X * c.Y;
        unsigned head = 0, tail = 1;
        int n = 0;
        {
            const int sz = div_by(start, c.magic_xy), srem = start - sz * XY;
            if (sz + 1 >= c.Z || !((c.col[srem] >> (sz + 1)) & 1u)) return 0;
        }
        if (lane == 0) {
            c.q_cl[0] = (uint32_t)start | (1u << 12);
            c.q_nj[0] = 0;
            if (PARENTS) c.q_par[0] = (uint16_t)start;
            c.best[start] = 1;
        }
        __syncwarp();
        const int dx = lane == 0 ? 1 : (lane == 2 ? -1 : 0);       // helper_3D.py:220 direction order
        const int dy = lane == 1 ? 1 : (lane == 3 ? -1 : 0);
        while (head != tail) {
            const uint32_t cl = c.q_cl[head & (MAZE_QCAP - 1)];
            const int nj_e = c.q_nj[head & (MAZE_QCAP - 1)];
            ++head;
            const int cell = cl & 0xFFF, ln = cl >> 12;
            const int z = div_by(cell, c.magic_xy), rem = cell - z * XY, y = div_by(rem, c.magic_x), x = rem - y * c.X;
            const uint16_t b = c.best[cell];
            const bool first = !(b & 0x8000u);
            if (lane == 0) {
                if (first) {
                    if (n < c.order_cap) c.order[n] = (uint16_t)cell;
                    c.best[cell] = b | 0x8000u;
                }
                c.nj[cell] = (uint16_t)nj_e;
                if (PARENTS) c.par[cell] = c.q_par[(head - 1) & (MAZE_QCAP - 1)];
            }
            n += first;
            bool valid = false;
            int ncell = 0, cost = 0, jump = 0;
            if (lane < 4) {
                valid = move(c, x, y, z, dx, dy, ncell, cost, jump);
                if (valid) {
                    const int nb = c.best[ncell] & 0x7FFF;
                    if (nb != 0 && nb <= ln + cost) valid = false;   // would be skipped at pop (:437-440)
                }
            }
            const unsigned m = __ballot_sync(0xffffffffu, valid);
            if (valid) {
                const unsigned pos = (tail + __popc(m & ((1u << lane) - 1u))) & (MAZE_QCAP - 1);
                c.q_cl[pos] = (uint32_t)ncell | ((uint32_t)(ln + cost) << 12);
                c.q_nj[pos] = (uint16_t)(nj_e + jump);
                if (PARENTS) c.q_par[pos] = (uint16_t)cell;
                c.best[ncell] = (uint16_t)((c.best[ncell] & 0x8000u) | (ln + cost));
            }
            tail += __popc(m);
            if (tail - head > (unsigned)MAZE_QCAP || n > c.order_cap) {
                overflow = true;
                break;
            }
            __syncwarp();
        }
        __syncwarp();
        return n < c.order_cap ? n : c.order_cap;
    }

    // first maximum of len(paths[.]) in insertion order (np.argmax, helper_3D.py:538-541)
    __device__ static __forceinline__ void far_tile(const Ctx& c, int n, int lane, int& cell, int& dist) {
        uint32_t key = 0;
        for (int i = lane; i < n; i += 32) {
            const uint32_t k = ((uint32_t)(c.best[c.order[i]] & 0x7FFF) << 16) | (uint32_t)(0xFFFF - i);
            key = max(key, k);
        }
        key = __reduce_max_sync(0xffffffffu, key);
        cell = c.order[0xFFFF - (key & 0xFFFF)];
        dist = key >> 16;
    }

    __device__ static __forceinline__ void clear_search(Ctx& c, int n, int lane) {
        for (int i = lane; i < n; i += 32) c.best[c.order[i]] = 0;
        __syncwarp();
    }

    __device__ static void stats(const KParams& p, Ctx& c, const int8_t* grid, int lane, int32_t* out) {
        const int Z = c.Z, Y = c.Y, X = c.X, R = c.R;
        // ---- stage the grid (coalesced 128-bit loads), build the row / column AIR masks --------------------
        {
            uint4* stage = (uint4*)c.best;
            const uint4* src = (const uint4*)grid;
            for (int i = lane; i < p.row_stride / 16; i += 32) stage[i] = src[i];
            __syncwarp();
            const uint8_t* g = (const uint8_t*)c.best;
            for (int r = lane; r < R; r += 32) {
                uint32_t m = 0;
                for (int x = 0; x < X; ++x) m |= (uint32_t)(g[r * X + x] == 0) << x;
                c.row[r] = (uint16_t)m;
            }
            for (int q = lane; q < Y * X; q += 32) {
                uint32_t m = 0;
                for (int z = 0; z < Z; ++z) m |= (uint32_t)(g[z * Y * X + q] == 0) << z;
                c.col[q] = (uint16_t)m;
            }
            __syncwarp();
            uint4* bz = (uint4*)c.best;
            for (int i = lane; i < c.best_bytes / 16; i += 32) bz[i] = make_uint4(0, 0, 0, 0);
            __syncwarp();
        }

        // ---- calc_longest_path (helper_3D.py:503-563) ---------------------------------------------------------
        int final_value = 0, last_far = -1;
        uint32_t planes = 0;
        bool overflow = false, index_error = false;
        for (int z = 1; z + 1 < Z; ++z) {
            if ((planes >> z) & 1u) continue;                                            // :515
            // start tiles of this plane: AIR with head-room (:520) standing on a solid tile (:525)
            uint32_t cand = 0;
            if (lane < Y) cand = c.row[z * Y + lane] & c.row[(z + 1) * Y + lane] & ~(uint32_t)c.row[(z - 1) * Y + lane];
            const unsigned rows_with = __ballot_sync(0xffffffffu, cand != 0);
            if (!rows_with) continue;
            const int y = __ffs(rows_with) - 1;
            const int x = __ffs(__shfl_sync(0xffffffffu, cand, y)) - 1;
            const int start = (z * Y + y) * X + x;

            int n = search(c, start, lane, overflow);                                    // :529
            uint32_t mark = 0;
            for (int i = lane; i < n; i += 32) {                                          // :531
                const int cell = c.order[i];
                const int cz = div_by(cell, c.magic_xy), rem = cell - cz * X * Y, cy = div_by(rem, c.magic_x),
                          cx = rem - cy * X;
                mark |= (1u << cx) | (1u << cy) | (1u << cz);
            }
            mark = __reduce_or_sync(0xffffffffu, mark);
            if (mark >> Z) index_error = true;
            planes |= mark;
            int far, dist;
            far_tile(c, n, lane, far, dist);                                             // :538-541
            clear_search(c, n, lane);
            n = search(c, far, lane, overflow);                                          // :548
            far_tile(c, n, lane, far, dist);                                             // :549-552
            last_far = far;                                                              // :553 last component wins
            if (dist > final_value) final_value = dist;                                  // :558
            clear_search(c, n, lane);
            if (overflow) break;
        }

        // ---- calc_num_regions (helper_3D.py:396-406): 6-neighbour AIR components by union-find over runs ---
        // (u32 run parents; u16 per-cell parents, count_regions_rows, ran at 2.12 against 2.26e7 env-steps/s on B200, 14^3)
        const int regions = count_regions_runs32(c.row, Z, Y, X, (uint32_t*)c.best, lane);

        if (lane == 0) {
            // jumps[far] of the last processed component: nj[] still holds that search's recordings (lane 0
            // wrote them, so its own load sees them)
            out[0] = regions;
            out[1] = final_value;
            out[2] = last_far >= 0 ? c.nj[last_far] : 0;
            if (p.status && (index_error || overflow)) atomicOr(p.status, (index_error ? 2 : 0) | (overflow ? 4 : 0));
        }
    }
};

}  // namespace pcgrl
