// minecraft_3D_holey_maze / minecraft_3D_dungeon_holey (SURVEY.md 8f rank 2): get_stats on the BORDERED map with an
// entrance and an exit (foot + head tile each) dug into the border, with minecraft_3D_maze's player search.
//
// Reference path replaced (paths relative to /root/reference/control_pcgrl/envs/):
//   probs/minecraft/minecraft_3D_holey_maze_prob.py:71-130     get_stats: one search from the entrance;
//       connected-path-length = len(path to the exit) or -1, n_jump = jumps on it, path-length = number of tiles of
//       the longest recorded path after remove_stacked_path_tiles (helper_3D.py:657-675) -- of the PREVIOUS call,
//       because :92-93 read self.path_coords before assigning it
//   probs/minecraft/minecraft_3D_holey_dungeon_prob.py:95-146  get_stats: chests / enemies counts, nearest-enemy =
//       shortest positive path length from the entrance to a SKULL / PUMPKIN, path-length / n_jump = entrance ->
//       first chest -> exit; the player walks through everything but DIRT, regions are counted over AIR only
//   probs/holey_prob_3D.py:16-100                               border cells, gen_holes, _valid_holes
//   helper_3D.py:422-490, 214-319                               run_dijkstra, _passable (maze3d_search.cuh)
//
// The level grid in HBM is the interior [Z, Y, X]; the kernel builds the bordered bit masks itself (border = DIRT,
// the four hole tiles = AIR).  pcgrl_state.holes holds (ez, ey, ex, xz, xy, xx): the FOOT tiles in bordered
// coordinates, the head tile is the one above -- except for the reference's "no valid exit found" default, an exit
// at (1, 1, 1) whose head is the same tile (holey_prob_3D.py:86, 94-98: exit_coords stays np.ones((2, 3))).
//
// The longest path itself is needed (its tile SET, de-stacked), not just its length: the search keeps a parent cell
// per recorded cell.  In the reference every queue entry carries its own path list; the final list of a cell equals
// the final list of its final parent plus the move's tiles, because a cell whose path gets shorter re-pushes all
// its moves and every child then re-records the shorter path (validated on the CPU against the reference's lists
// and pinned on tests/golden/stats_maze3d_holey.npz).
#include "maze3d_search.cuh"

namespace pcgrl {

template <bool DUNGEON>
struct Holey3DProb {
    static constexpr int K = DUNGEON ? 6 : 5;
    // maze:    regions, path-length (of the previous call), connected-path-length, n_jump, _next-path-length
    // dungeon: regions, path-length, chests, enemies, nearest-enemy, n_jump
    using Ctx = Maze3DProb::Ctx;

    __device__ static Ctx make_ctx(const KParams& p, uint8_t* ws, int global_warp) {
        return Maze3DProb::make_ctx_dims(p, ws, global_warp, p.d0 + 2, p.d1 + 2, p.d2 + 2);
    }
    __device__ static __forceinline__ int bcell(const Ctx& c, int z, int y, int x) { return (z * c.Y + y) * c.X + x; }
    __device__ static __forceinline__ void dig(Ctx& c, int z, int y, int x) {   // lane 0
        c.col[y * c.X + x] |= (uint16_t)(1u << z);
        c.row[z * c.Y + y] |= (uint16_t)(1u << x);
    }

    __device__ static void stats(const KParams& p, Ctx& c, const int8_t* grid, int lane, int32_t* out) {
        const int Z = c.Z, Y = c.Y, X = c.X, R = c.R;
        const int iZ = p.d0, iY = p.d1, iX = p.d2;
        const int64_t idx = (grid - (p.mode == MODE_STATS ? p.stats_grids : p.grids)) / p.row_stride;
        const int hs = (!DUNGEON && p.mode == MODE_STATS) ? 7 : 6;    // pcgrl_stats_holey carries the previous length
        const int32_t* h = p.holes + idx * hs;
        // ---- stage the interior grid; bordered masks: col = what the player walks through, row = AIR (regions) ----
        int n_chest = 0, n_enemy = 0, first_chest = 0x7FFFFFFF;
        {
            uint4* stage = (uint4*)c.best;
            const uint4* src = (const uint4*)grid;
            for (int i = lane; i < p.row_stride / 16; i += 32) stage[i] = src[i];
            __syncwarp();
            const uint8_t* g = (const uint8_t*)c.best;
            for (int r = lane; r < R; r += 32) {          // r = zb * Y + yb
                const int zb = r / Y, yb = r - zb * Y;
                uint32_t m = 0;
                if (zb >= 1 && zb <= iZ && yb >= 1 && yb <= iY)
                    for (int x = 0; x < iX; ++x) m |= (uint32_t)(g[((zb - 1) * iY + (yb - 1)) * iX + x] == 0) << (x + 1);
                c.row[r] = (uint16_t)m;
            }
            for (int q = lane; q < Y * X; q += 32) {      // q = yb * X + xb
                const int yb = q / X, xb = q - yb * X;
                uint32_t m = 0;
                if (yb >= 1 && yb <= iY && xb >= 1 && xb <= iX)
                    for (int z = 0; z < iZ; ++z) {
                        const int t = g[(z * iY + (yb - 1)) * iX + (xb - 1)];
                        m |= (uint32_t)(DUNGEON ? t != 1 : t == 0) << (z + 1);
                    }
                c.col[q] = (uint16_t)m;
            }
            if (DUNGEON) {
                for (int i = lane; i < p.cells; i += 32) {
                    const int t = g[i];
                    n_chest += t == 2;
                    n_enemy += t == 3 || t == 4;
                    if (t == 2) first_chest = min(first_chest, i);   // get_tile_locations scans z, y, x (helper_3D.py:22-29)
                }
                n_chest = __reduce_add_sync(0xffffffffu, n_chest);
                n_enemy = __reduce_add_sync(0xffffffffu, n_enemy);
                first_chest = __reduce_min_sync(0xffffffffu, first_chest);
            }
            __syncwarp();
            if (lane == 0) {     // the holes: foot and head of the entrance and of the exit become AIR
                dig(c, h[0], h[1], h[2]);
                dig(c, h[0] + 1, h[1], h[2]);
                dig(c, h[3], h[4], h[5]);
                if (!(h[3] == 1 && h[4] == 1 && h[5] == 1)) dig(c, h[3] + 1, h[4], h[5]);
            }
            __syncwarp();
        }
        const int entrance = bcell(c, h[0], h[1], h[2]), exit_c = bcell(c, h[3], h[4], h[5]);
        bool overflow = false;
        int v1 = 0, v2 = 0, v3 = 0, v4 = 0;     // problem-specific outputs, see below
        if (!DUNGEON) {
            // the enemy / chest scan above read the staged grid out of c.best: clear it for the search
            uint4* bz = (uint4*)c.best;
            for (int i = lane; i < c.best_bytes / 16; i += 32) bz[i] = make_uint4(0, 0, 0, 0);
            __syncwarp();
            const int n = Maze3DProb::search<true>(c, entrance, lane, overflow);                             // :81
            const uint16_t bx = c.best[exit_c];
            v2 = (bx & 0x8000u) ? (bx & 0x7FFF) : -1;                                            // :84 connected-path-length
            v3 = 0;
            if (lane == 0 && (bx & 0x8000u)) v3 = c.nj[exit_c];                                   // :89 n_jump
            v3 = __shfl_sync(0xffffffffu, v3, 0);
            int far = entrance, dist = 0;
            if (n > 0) Maze3DProb::far_tile(c, n, lane, far, dist);                               // :90-92 first longest path
            // its tile set (path tiles + the tiles each move passes through), as one z-mask per column
            uint16_t* colset = c.q_nj;       // the FIFO is empty now: 2 * MAZE_QCAP bytes >= Y * X masks
            for (int q = lane; q < Y * X; q += 32) colset[q] = 0;
            __syncwarp();
            if (lane == 0 && n > 0) {
                const int XY = X * Y;
                int cell = far;
                for (int guard = 0; guard < c.cells; ++guard) {
                    const int cz = cell / XY, cr = cell - cz * XY, cy = cr / X, cx = cr - cy * X;
                    colset[cy * X + cx] |= (uint16_t)(1u << cz);
                    const int par = c.par[cell];
                    if (par == cell) break;
                    const int pz = par / XY, pr = par - pz * XY, py = pr / X, px = pr - py * X;
                    const int mx = (px + cx) / 2, my = (py + cy) / 2;          // the gap tile of a jump
                    if (abs(cx - px) + abs(cy - py) == 2) {                     // jumps pass over (mx, my)
                        colset[my * X + mx] |= (uint16_t)(1u << pz);
                        if (cz != pz) colset[my * X + mx] |= (uint16_t)(1u << cz);   // up: (m, z + 1); down: (m, z - 1)
                    } else if (cz == pz - 1) {
                        colset[cy * X + cx] |= (uint16_t)(1u << pz);            // step down: through (n, z)
                    } else if (cz == pz + 1) {
                        colset[py * X + px] |= (uint16_t)(1u << cz);            // step up: through (x, y, z + 1)
                    }
                    cell = par;
                }
            }
            __syncwarp();
            int kept = 0;                                                        // remove_stacked_path_tiles (:94)
            for (int q = lane; q < Y * X; q += 32) {
                const uint32_t m = colset[q];
                kept += __popc(m & ~(m << 1));
            }
            v4 = __reduce_add_sync(0xffffffffu, kept);
            // path-length reports the length found by the PREVIOUS call (:92-93)
            v1 = p.mode == MODE_STATS ? h[6] : p.stats[idx * K + 4];
            Maze3DProb::clear_search(c, n, lane);
        } else {
            uint4* bz = (uint4*)c.best;
            for (int i = lane; i < c.best_bytes / 16; i += 32) bz[i] = make_uint4(0, 0, 0, 0);
            __syncwarp();
            int path = 0, nj = 0, nearest = 0;
            if (n_enemy > 0 || n_chest > 0) {
                const int n = Maze3DProb::search<false>(c, entrance, lane, overflow);                       // :113 / :131
                if (n_enemy > 0) {                                                               // :114-124
                    // enemy cells are found again in the grid in HBM (the stage was cleared for the search)
                    uint32_t best = 0xFFFFFFFFu;
                    for (int i = lane; i < p.cells; i += 32) {
                        const int t = grid[i];
                        if (t == 3 || t == 4) {
                            const int z = i / (iY * iX), r = i - z * iY * iX, y = r / iX, x = r - y * iX;
                            const uint16_t b = c.best[bcell(c, z + 1, y + 1, x + 1)];
                            if ((b & 0x8000u) && (b & 0x7FFF) > 0) best = min(best, (uint32_t)(b & 0x7FFF));
                        }
                    }
                    best = __reduce_min_sync(0xffffffffu, best);
                    nearest = best == 0xFFFFFFFFu ? 0 : (int)best;
                }
                int chest = -1;
                if (n_chest > 0) {                                                               // :127-135
                    const int z = first_chest / (iY * iX), r = first_chest - z * iY * iX, y = r / iX, x = r - y * iX;
                    chest = bcell(c, z + 1, y + 1, x + 1);
                    const uint16_t b = c.best[chest];
                    if (b & 0x8000u) {
                        path += b & 0x7FFF;
                        int j = 0;
                        if (lane == 0) j = c.nj[chest];
                        nj += __shfl_sync(0xffffffffu, j, 0);
                    }
                }
                Maze3DProb::clear_search(c, n, lane);
                if (chest >= 0) {                                                                // :137-141
                    const int n2 = Maze3DProb::search<false>(c, chest, lane, overflow);
                    const uint16_t b = c.best[exit_c];
                    if (b & 0x8000u) {
                        path += b & 0x7FFF;
                        int j = 0;
                        if (lane == 0) j = c.nj[exit_c];
                        nj += __shfl_sync(0xffffffffu, j, 0);
                    }
                    Maze3DProb::clear_search(c, n2, lane);
                }
            }
            v1 = path;
            v2 = nearest;
            v3 = nj;
        }
        // ---- calc_num_regions over AIR of the bordered map (helper_3D.py:396-406) ----------------------------------
        const int regions = count_regions_runs32(c.row, Z, Y, X, (uint32_t*)c.best, lane);
        if (lane == 0) {
            out[0] = regions;
            if (!DUNGEON) {
                out[1] = v1;
                out[2] = v2;
                out[3] = v3;
                out[4] = v4;
            } else {
                out[1] = v1;
                out[2] = n_chest;
                out[3] = n_enemy;
                out[4] = v2;
                out[5] = v3;
            }
            if (p.status && overflow) atomicOr(p.status, 4);
        }
    }
};

cudaError_t launch_maze3d_holey(const KParams& p, int problem, cudaStream_t s, bool& supported) {
    // the bordered map must fit the 16-bit masks
    supported = p.ndim == 3 && p.d0 <= 14 && p.d1 <= 14 && p.d2 <= 14 && p.d0 >= 3 && p.scratch != nullptr && p.holes != nullptr;
    if (!supported) return cudaSuccess;
    const MazeLayout L = maze_layout(p.d0 + 2, p.d1 + 2, p.d2 + 2, p.row_stride);
    if (problem == PCGRL_PROB_MINECRAFT_3D_HOLEY_MAZE)
        return launch_search<Holey3DProb<false>, MAZE_WARPS>(p, s, L.total, MAZE_CTAS_PER_SM, MAZE_MAX_CTAS);
    return launch_search<Holey3DProb<true>, MAZE_WARPS>(p, s, L.total, MAZE_CTAS_PER_SM, MAZE_MAX_CTAS);
}

}  // namespace pcgrl
