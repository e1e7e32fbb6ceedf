// Env-step pieces shared by every step kernel (bit-board and search problems): the representation update,
// episode reset, and the thread-per-env phases A (action, counters, change flag) and D (reward, outputs).
#pragma once
#include "pcgrl_device.cuh"

namespace pcgrl {

// ------------------------------------------------------------------------------------------------
// phase A helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int cell_index(const KParams& p, int a0, int a1, int a2) {
    return (a0 * p.d1 + a1) * p.d2 + a2;
}

// Apply one non-cellular action to env `gid`; updates pos / n_step in HBM.
// Returns bit0 = change (what PcgrlEnv counts in _changes), bit1 = the grid was actually modified.  The two
// differ only under StaticTileRepresentation (envs/reps/wrappers.py:358-376): an edit of a frozen cell is
// undone (`np.where(static_tiles < 1, new, old)`), but `change = np.any(old_state != new_state)` compares
// against the pre-undo array, so it still counts as a change (and the reference recomputes identical stats).
// *cell_out (optional): linear index of the one cell the action addressed, -1 for multi-cell actions (patch).
__device__ __forceinline__ int apply_action(const KParams& p, int64_t gid, int* cell_out = nullptr) {
    int8_t* grid = p.grids + gid * p.row_stride;
    int32_t* pos = p.pos + gid * 3;
    const uint8_t* frozen = p.static_mask ? p.static_mask + gid * p.row_stride : nullptr;
    int change = 0, wrote = 0;
    if (cell_out) *cell_out = -1;
    if (p.rep == PCGRL_REP_NARROW && p.action_kind == PCGRL_ACT_PATCH) {
        // MultiActionRepresentation.update (envs/reps/wrappers.py:466-528): the patch action.reshape(act_window)
        // replaces map[pos - l_pad : pos + r_pad + 1], l_pad = floor((a-1)/2), r_pad = ceil((a-1)/2) (:404-411);
        // change = any cell differs; then pos = act_coords[n_step % len], n_step += 1 (:517-518)
        const int np_ = p.aw0 * p.aw1 * p.aw2;
        const int32_t* a = (const int32_t*)p.actions + gid * np_;
        const int l0 = (p.aw0 - 1) / 2, l1 = (p.aw1 - 1) / 2, l2 = (p.aw2 - 1) / 2;
        const int t0 = pos[0] - l0, t1 = pos[1] - l1, t2 = pos[2] - l2;
        if (t0 < 0 || t1 < 0 || t2 < 0 || t0 + p.aw0 > p.d0 || t1 + p.aw1 > p.d1 || t2 + p.aw2 > p.d2) {
            if (p.status) atomicOr(p.status, 1);   // the reference asserts the patch lies inside the map (:498-501)
        } else {
            int idx = 0;
            for (int i0 = 0; i0 < p.aw0; ++i0)
                for (int i1 = 0; i1 < p.aw1; ++i1)
                    for (int i2 = 0; i2 < p.aw2; ++i2, ++idx) {
                        const int v = a[idx];
                        if ((unsigned)v >= (unsigned)p.n_tiles) {
                            if (p.status) atomicOr(p.status, 1);
                            continue;
                        }
                        const int c = cell_index(p, t0 + i0, t1 + i1, t2 + i2);
                        if (grid[c] != v) {
                            change = 1;
                            if (!frozen || !frozen[c]) {
                                grid[c] = (int8_t)v;
                                wrote = 1;
                            }
                        }
                    }
        }
        // get_act_coords (:445-463): np.meshgrid(*ranges).T.reshape(-1, ndim) -- row-major in 2D; in 3D the
        // LAST axis is the slowest, then axis 0, then axis 1 (meshgrid's 'xy' indexing swaps the first two)
        const int n0 = p.d0 - p.aw0 + 1, n1 = p.d1 - p.aw1 + 1, n2 = p.d2 - p.aw2 + 1;
        const int ns = p.n_step[gid];
        const int k = ns % (n0 * n1 * n2);
        pos[1] = l1 + k % n1;
        pos[0] = l0 + (k / n1) % n0;
        pos[2] = l2 + k / (n1 * n0);
        p.n_step[gid] = ns + 1;
    } else if (p.rep == PCGRL_REP_NARROW) {
        // reps/narrow_rep.py:89-102: write at _pos, then _pos = coords[n_step % N], then n_step += 1
        const int a = load_action(p, gid);
        const int c = cell_index(p, pos[0], pos[1], pos[2]);
        if (cell_out) *cell_out = c;
        if ((unsigned)a >= (unsigned)p.n_tiles) {
            if (p.status) atomicOr(p.status, 1);
        } else {
            const int old = grid[c];
            change = old != a;
            wrote = change && !(frozen && frozen[c]);
            if (wrote) grid[c] = (int8_t)a;
        }
        const int ns = p.n_step[gid];
        const int k = ns % p.cells;
        pos[2] = k % p.d2;
        pos[1] = (k / p.d2) % p.d1;
        pos[0] = k / (p.d2 * p.d1);
        p.n_step[gid] = ns + 1;
    } else if (p.rep == PCGRL_REP_TURTLE) {
        // reps/turtle_rep.py:87-107: 0..3 move along axis 0 / axis 1 (clamped), >= 4 writes tile a-4
        const int a = load_action(p, gid);
        if (a >= 0 && a < 4) {
            const int axis = a >> 1;
            const int lim = (axis == 0 ? p.d0 : p.d1) - 1;
            int v = pos[axis] + ((a & 1) ? 1 : -1);
            pos[axis] = v < 0 ? 0 : (v > lim ? lim : v);
        } else if (a >= 4 && a - 4 < p.n_tiles) {
            const int c = cell_index(p, pos[0], pos[1], pos[2]);
            if (cell_out) *cell_out = c;
            const int t = a - 4;
            const int old = grid[c];
            change = old != t;
            wrote = change && !(frozen && frozen[c]);
            if (wrote) grid[c] = (int8_t)t;
        } else if (p.status) {
            atomicOr(p.status, 1);
        }
    } else {  // PCGRL_REP_WIDE
        int q0, q1, q2 = 0, v;
        if (p.action_kind == PCGRL_ACT_WIDE_FLAT) {
            // wrappers.py:304-323: (y, x, v) = unravel(a, (h, w, C)); env.step([x, y, v]) -> _map[x, y] = v
            const int a = load_action(p, gid);
            v = a % p.n_tiles;
            const int x = (a / p.n_tiles) % p.act_w;
            const int y = a / (p.n_tiles * p.act_w);
            q0 = x;
            q1 = y;
            if (a < 0 || y >= p.act_h) q0 = -1;
        } else {
            const int32_t* a = (const int32_t*)p.actions + gid * (p.ndim + 1);
            q0 = a[0];
            q1 = a[1];
            if (p.ndim == 3) q2 = a[2];
            v = a[p.ndim];
        }
        if ((unsigned)q0 >= (unsigned)p.d0 || (unsigned)q1 >= (unsigned)p.d1 || (unsigned)q2 >= (unsigned)p.d2 ||
            (unsigned)v >= (unsigned)p.n_tiles) {
            if (p.status) atomicOr(p.status, 1);
        } else {
            const int c = cell_index(p, q0, q1, q2);
            if (cell_out) *cell_out = c;
            const int old = grid[c];
            change = old != v;
            wrote = change;   // the reference's wide / cellular reps do not run under StaticTileRepresentation
            if (change) grid[c] = (int8_t)v;
            pos[0] = q0;
            pos[1] = q1;
            pos[2] = q2;
        }
    }
    return change | (wrote << 1);
}

// HoleyProblem.gen_holes (envs/probs/holey_prob.py:32-60) for a 2D map.  Border cells are numbered in the
// row-major order of get_border_idxs (:20-30): the top row (x = 1..W), then (y, 0), (y, W+1) for y = 1..H, then
// the bottom row.
__device__ __forceinline__ void border_cell(int k, int H, int W, int& y, int& x) {
    if (k < W) {
        y = 0;
        x = 1 + k;
    } else if (k < W + 2 * H) {
        const int j = k - W;
        y = 1 + (j >> 1);
        x = (j & 1) ? W + 1 : 0;
    } else {
        y = H + 1;
        x = 1 + (k - W - 2 * H);
    }
}
// _valid_holes (:74-90), restated literally: the reference names the pair (x, y) although coords[0] is the row,
// and compares with _width - 1 / _height - 1 although the bordered map is two cells larger.
__device__ __forceinline__ bool valid_holes(int a0, int a1, int b0, int b1, int H, int W) {
    auto pull = [&](int& x, int& y) {
        if (x == 0) x = 1;
        else if (x == W - 1) x = W - 2;
        else if (y == 0) y = 1;
        else if (y == H - 1) y = H - 2;
    };
    pull(a0, a1);
    pull(b0, b1);
    return max(abs(a0 - b0), abs(a1 - b1)) > 1;
}
__device__ static void gen_holes(const KParams& p, int64_t gid, uint64_t genv, uint2 key) {
    int32_t* h = p.holes + gid * 4;
    const int H = p.d0, W = p.d1;
    if (p.hole_mode == PCGRL_HOLES_FIXED) {   // :47-49 entrance (1, 0); exit np.array((_width, _height + 1))
        h[0] = 1;
        h[1] = 0;
        h[2] = W;
        h[3] = H + 1;
        return;
    }
    // np.random.choice(n_border, size=4, replace=False): four distinct cells by rejection (Philox; the
    // reference's global numpy stream is not part of the parity contract)
    const int nb = 2 * (H + W);
    int pick[4], n = 0;
    for (uint32_t c = 0; n < 4 && c < 16; ++c) {
        const uint4 r = philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)p.epoch, 0xD0000000u + c), key);
        const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
        for (int j = 0; j < 4 && n < 4; ++j) {
            const int k = (int)(rr[j] % (uint32_t)nb);
            bool dup = false;
            for (int q = 0; q < n; ++q) dup |= pick[q] == k;
            if (!dup) pick[n++] = k;
        }
    }
    int ey, ex;
    border_cell(pick[0], H, W, ey, ex);
    h[0] = ey;
    h[1] = ex;
    for (int i = 1; i < n; ++i) {
        int y, x;
        border_cell(pick[i], H, W, y, x);
        if (valid_holes(ey, ex, y, x, H, W)) {
            h[2] = y;
            h[3] = x;
            return;
        }
    }
    // no candidate accepted: the reference keeps the exit of the previous episode (:53-58); a first episode
    // (exit never set: both coordinates 0, a corner no hole can occupy) falls back to the fixed exit
    if (h[2] == 0 && h[3] == 0) {
        h[2] = W;
        h[3] = H + 1;
    }
}

// HoleyProblem3D.gen_holes (envs/probs/holey_prob_3D.py:41-100): holes[gid] = (ez, ey, ex, xz, xy, xx), the foot tiles
// in bordered coordinates.  Border cells (get_border_idxs, :16-35): the four side faces without their vertical
// edges, z = 1 .. Z - 1 (the reference's `1:-2` leaves the top interior layer out), in argwhere order z, y, x.
__device__ static void gen_holes3d(const KParams& p, int64_t gid, uint64_t genv, uint2 key) {
    int32_t* h = p.holes + gid * 6;
    const int Z = p.d0, Y = p.d1, X = p.d2;
    if (p.hole_mode == PCGRL_HOLES_FIXED) {    // :66-69 diagonal corners
        h[0] = 1, h[1] = 0, h[2] = X;
        h[3] = 2, h[4] = Y + 1, h[5] = 1;
        return;
    }
    const int per = 2 * (Y + X), nb = (Z - 1) * per;
    const int want = nb < 26 ? nb : 26;        // :74-75 `potential` distinct random border cells
    int pick[26], n = 0;
    for (uint32_t c = 0; n < want && c < 64; ++c) {
        const uint4 r = philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)p.epoch, 0xD0000000u + c), key);
        const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
        for (int j = 0; j < 4 && n < want; ++j) {
            const int k = (int)(rr[j] % (uint32_t)nb);
            bool dup = false;
            for (int q = 0; q < n; ++q) dup |= pick[q] == k;
            if (!dup) pick[n++] = k;
        }
    }
    auto cell = [&](int k, int& z, int& y, int& x) {
        z = 1 + k / per;
        border_cell(k % per, Y, X, y, x);
    };
    int ez = 1, ey = 0, ex = 1;
    if (n > 0) cell(pick[0], ez, ey, ex);
    h[0] = ez, h[1] = ey, h[2] = ex;
    h[3] = h[4] = h[5] = 1;                    // :86 exit_coords = np.ones((2, 3)) when no candidate is accepted
    for (int i = 1; i < n; ++i) {
        int z, y, x;
        cell(pick[i], z, y, x);
        // _valid_holes (:96-100): np.max over |foot - xyz| and |head - xyz|, all three coordinates
        const int d = max(max(max(abs(ez - z), abs(ez + 1 - z)), abs(ey - y)), abs(ex - x));
        if (d > 1) {
            h[3] = z, h[4] = y, h[5] = x;
            break;
        }
    }
}

// Episode start for env `gid` (thread-per-env): grid from src or Philox, counters, start position.
__device__ static void reset_env(const KParams& p, int64_t gid) {
    int8_t* grid = p.grids + gid * p.row_stride;
    const uint64_t genv = (uint64_t)(p.env_offset + gid);
    const uint2 key = make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32));
    if (p.src_grids) {
        const uint4* s = (const uint4*)(p.src_grids + gid * p.row_stride);
        uint4* d = (uint4*)grid;
        for (int i = 0; i < p.row_stride / 16; ++i) d[i] = s[i];
    } else {
        float cdf[PCGRL_MAX_TILES];
        if (p.init_random_probs) {
            // pcgrl_env.py:162-164 + helper.get_int_prob: per-episode tile probabilities U(0,1)^C, normalised
            float tot = 0.f;
            for (int t0 = 0; t0 < p.n_tiles; t0 += 4) {
                const uint4 r = philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)p.epoch,
                                                         0x80000000u + t0), key);
                const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
                for (int j = 0; j < 4 && t0 + j < p.n_tiles; ++j) {
                    tot += u01(rr[j]) + 1e-7f;
                    cdf[t0 + j] = tot;
                }
            }
            for (int t = 0; t < p.n_tiles; ++t) cdf[t] /= tot;
        } else {
            for (int t = 0; t < p.n_tiles; ++t) cdf[t] = p.init_cdf[t];
        }
        for (int c0 = 0; c0 < p.row_stride; c0 += 16) {
            uint32_t w[4] = {0, 0, 0, 0};
            for (int q = 0; q < 4; ++q) {
                const uint4 r = philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)p.epoch,
                                                         (uint32_t)(c0 / 4 + q)), key);
                const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
                for (int j = 0; j < 4; ++j) {
                    const int c = c0 + q * 4 + j;
                    int t = 0;
                    if (c < p.cells) {
                        const float u = u01(rr[j]);
                        while (t < p.n_tiles - 1 && u >= cdf[t]) ++t;
                    }
                    w[q] |= (uint32_t)t << (8 * j);
                }
            }
            *(uint4*)(grid + c0) = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
    if (!p.src_grids && p.static_mask && (p.static_prob > 0.f || p.n_static_walls > 0)) {
        // StaticTileRepresentation.reset (envs/reps/wrappers.py:275-312).  Only the random-reset generator: with
        // caller-supplied maps the caller owns the mask (the reference's RNG stream is not part of the contract).
        uint8_t* sm = p.static_mask + gid * p.row_stride;
        float ps = 0.f;
        if (p.static_prob > 0.f) {   // :279-289 per-episode probability U(0,1) * static_prob (or fixed when evaluating)
            const uint4 r = philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)p.epoch, 0xB0000000u), key);
            ps = p.static_eval_mode ? p.static_prob : u01(r.x) * p.static_prob;
        }
        for (int c0 = 0; c0 < p.row_stride; c0 += 16) {
            uint32_t w[4] = {0, 0, 0, 0};
            if (ps > 0.f)
                for (int q = 0; q < 4; ++q) {
                    const uint4 r = philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)p.epoch,
                                                             0x40000000u + (uint32_t)(c0 / 4 + q)), key);
                    const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
                    for (int j = 0; j < 4; ++j)
                        if (c0 + q * 4 + j < p.cells && u01(rr[j]) < ps) w[q] |= 1u << (8 * j);
                }
            *(uint4*)(sm + c0) = make_uint4(w[0], w[1], w[2], w[3]);
        }
        // :291-308 random wall segments.  Restated with the reference's indexing: every start coordinate is drawn
        // from the length of the wall's own axis, the frozen cells are wall_pos in BORDERED coordinates (= map
        // coordinates wall_pos - 1) while the wall tiles are written to _map at wall_pos itself, i.e. one cell
        // further along every axis; numpy slicing clips whatever falls outside.
        const int dims[3] = {p.d0, p.d1, p.d2};
        for (int wi = 0; wi < p.n_static_walls; ++wi) {
            const uint4 r = philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)p.epoch,
                                                     0xA0000000u + 2u * wi), key);
            const uint4 r2 = philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)p.epoch,
                                                      0xA0000001u + 2u * wi), key);
            const int dim = (int)(r.x % (uint32_t)p.ndim);
            const int L = dims[dim];
            if (L < 3) continue;   // integers(1, L - 1) needs L >= 3
            const int len = 1 + (int)(r.y % (uint32_t)(L - 2));
            int wp[3] = {(int)(r.z % (uint32_t)L), (int)(r.w % (uint32_t)L), (int)(r2.x % (uint32_t)L)};
            wp[dim] = (int)(r2.y % (uint32_t)(L - len));
            if (p.ndim == 2) wp[2] = 0;
            for (int i = 0; i < len; ++i) {
                int m[3] = {wp[0], wp[1], wp[2]};
                m[dim] += i;
                if (m[0] < p.d0 && m[1] < p.d1 && m[2] < p.d2) sm[cell_index(p, m[0], m[1], m[2])] = 1;
                const int t0 = m[0] + 1, t1 = m[1] + 1, t2 = p.ndim == 3 ? m[2] + 1 : 0;
                if (t0 < p.d0 && t1 < p.d1 && t2 < p.d2) grid[cell_index(p, t0, t1, t2)] = (int8_t)p.wall_tile;
            }
        }
    }
    if (p.holes && p.hole_mode != PCGRL_HOLES_GIVEN) {
        if (p.ndim == 3) gen_holes3d(p, gid, genv, key);
        else gen_holes(p, gid, genv, key);
    }
    int32_t* pos = p.pos + gid * 3;
    pos[0] = pos[1] = pos[2] = 0;
    if (p.rep == PCGRL_REP_NARROW && p.action_kind == PCGRL_ACT_PATCH) {
        // the scan starts at act_coords[0] = the inner left pads (envs/reps/wrappers.py:404-411, 445-463)
        pos[0] = (p.aw0 - 1) / 2;
        pos[1] = (p.aw1 - 1) / 2;
        pos[2] = (p.aw2 - 1) / 2;
    }
    if (p.src_pos) {
        pos[0] = p.src_pos[gid * 3 + 0];
        pos[1] = p.src_pos[gid * 3 + 1];
        pos[2] = p.src_pos[gid * 3 + 2];
    } else if (p.rep == PCGRL_REP_TURTLE) {
        // reps/turtle_rep.py:41-44: int(random() * dim) per axis
        const uint4 r = philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)p.epoch, 0xC0000000u), key);
        pos[0] = min((int)(u01(r.x) * p.d0), p.d0 - 1);
        pos[1] = min((int)(u01(r.y) * p.d1), p.d1 - 1);
        if (p.ndim == 3) pos[2] = min((int)(u01(r.z) * p.d2), p.d2 - 1);
    }
    p.n_step[gid] = 0;
    p.iteration[gid] = 0;
    p.changes[gid] = 0;
    // reward / done are step outputs: an auto-reset must not erase the finishing step's values
}


// PcgrlEnv.step's bookkeeping for env `gid` after its representation update returned `cw` (bit0 change, bit1 the
// grid was modified): iteration / changes counters, done, change flag, zero reward for an unchanged map.
// Returns true when the stats must be recomputed (pcgrl_env.py:314).
__device__ __forceinline__ bool step_counters(const KParams& p, int64_t gid, int cw) {
    const int change = cw & 1;
    const int it = p.iteration[gid] + 1;   // pcgrl_env.py:279
    const int ch = p.changes[gid] + change;
    p.iteration[gid] = it;
    if (change) p.changes[gid] = ch;
    bool done = it > p.max_iterations;     // :307
    if (p.max_changes >= 0) done = done || ch > p.max_changes;  // :308-309
    p.done[gid] = done;
    if (p.changed) p.changed[gid] = change != 0;
    record_flags(p, gid, done, change);
    const bool need = (cw & 2) != 0;       // :314 stats only when the map changed (an undone edit of a frozen
                                           // tile leaves map, stats and loss as they were)
    if (!need) {
        p.reward[gid] = 0.f;
        record_reward(p, gid, 0.f);
    }
    return need;
}

// Phase D for one env: reward = loss(new stats) - loss(old stats) in fp64 (or the range-reward sum), then the new
// stats replace the old ones (int32 view and packed record).
// `old` (optional): the stats the reward is measured from, when p.stats no longer holds them (sokoban's deferred
// solver jobs: the step kernel already stored provisional stats there).
template <int K>
__device__ __forceinline__ void finish_env(const KParams& p, int64_t gid, const int32_t (&nw)[K],
                                           const int32_t* old = nullptr) {
    int32_t* st = p.stats + gid * K;
    if (p.mode == MODE_STEP) {
        int32_t od[K];
#pragma unroll
        for (int k = 0; k < K; ++k) od[k] = old ? old[k] : st[k];
        const double* trg = p.targets + (p.targets_per_env ? gid * K * 2 : 0);
        const double r = p.reward_mode == PCGRL_REWARD_RANGE
                             ? range_reward_sum(nw, od, trg, p.weights, K)
                             : control_loss(nw, trg, p.weights, K) - control_loss(od, trg, p.weights, K);
        p.reward[gid] = (float)r;
        record_reward(p, gid, (float)r);
    }
    record_stats<K>(p, gid, nw);
#pragma unroll
    for (int k = 0; k < K; ++k) st[k] = nw[k];
}

// ------------------------------------------------------------------------------------------------
// Cellular representation update (reps/ca_rep.py:31-44) of the tile_n envs starting at `base`, cooperative over
// the CTA: the whole map is replaced by the action.  s_flag[e] = 1 when env base + e's grid changed; the caller
// zeroes s_flag[0 .. tile_n) before.  Shared by the step kernels (phase_a) and k_update.  Ends with a __syncthreads().
// ------------------------------------------------------------------------------------------------
template <int THREADS>
__device__ __forceinline__ void cellular_rewrite(const KParams& p, int64_t base, int tile_n, uint8_t* s_flag) {
    const int tid = threadIdx.x;
    if (p.action_kind == PCGRL_ACT_CA_TILES) {
        const int chunks = p.row_stride / 16;
        for (int i = tid; i < tile_n * chunks; i += THREADS) {
            const int e = i / chunks, c = i - e * chunks;
            const int64_t off = (base + e) * p.row_stride + c * 16;
            const uint4 nw = *(const uint4*)((const int8_t*)p.actions + off);
            uint4* dst = (uint4*)(p.grids + off);
            const uint4 od = *dst;
            if (nw.x != od.x || nw.y != od.y || nw.z != od.z || nw.w != od.w) {
                *dst = nw;
                s_flag[e] = 1;
            }
        }
    } else if (p.cells % 4 == 0 && ((uintptr_t)p.actions & 15) == 0) {
        // PCGRL_ACT_CA_LOGITS, four cells per item: one 16-byte load per channel and one 4-byte grid word, so that a
        // thread keeps C x 16 bytes in flight instead of C x 4 (the rewrite streams the logits once: HBM-bound)
        const int q = p.cells / 4;
        for (int i = tid; i < tile_n * q; i += THREADS) {
            const int e = i / q, c = i - e * q;
            const float4* lg = (const float4*)p.actions + (base + e) * (int64_t)p.n_tiles * q + c;
            float4 best = __ldg(lg);
            int b0 = 0, b1 = 0, b2 = 0, b3 = 0;
            for (int t = 1; t < p.n_tiles; ++t) {   // strict > : ties keep the lowest channel
                const float4 v = __ldg(lg + (int64_t)t * q);
                if (v.x > best.x) best.x = v.x, b0 = t;
                if (v.y > best.y) best.y = v.y, b1 = t;
                if (v.z > best.z) best.z = v.z, b2 = t;
                if (v.w > best.w) best.w = v.w, b3 = t;
            }
            const uint32_t nw = (uint32_t)b0 | ((uint32_t)b1 << 8) | ((uint32_t)b2 << 16) | ((uint32_t)b3 << 24);
            uint32_t* g = (uint32_t*)(p.grids + (base + e) * p.row_stride) + c;
            if (*g != nw) {
                *g = nw;
                s_flag[e] = 1;
            }
        }
    } else {  // PCGRL_ACT_CA_LOGITS: float32 [N, C, cells]; argmax over C, ties -> lowest index
        for (int i = tid; i < tile_n * p.cells; i += THREADS) {
            const int e = i / p.cells, c = i - e * p.cells;
            const float* lg = (const float*)p.actions + (base + e) * (int64_t)p.n_tiles * p.cells + c;
            float best = lg[0];
            int bi = 0;
            for (int t = 1; t < p.n_tiles; ++t) {
                const float v = lg[(int64_t)t * p.cells];
                if (v > best) {
                    best = v;
                    bi = t;
                }
            }
            int8_t* g = p.grids + (base + e) * p.row_stride + c;
            if (*g != bi) {
                *g = (int8_t)bi;
                s_flag[e] = 1;
            }
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// phase A (whole CTA): apply the actions of the TILE envs starting at `base` (or reset them, or just list
// them in MODE_STATS), advance the counters, decide done, and build the compact list of envs whose map
// changed -- only those need get_stats (pcgrl_env.py:314).
//   s_list[slot] = tile-local env index, s_slot[env] = slot or -1, s_flag = scratch, *s_count = #listed.
// Ends with a __syncthreads().
// ------------------------------------------------------------------------------------------------
template <int THREADS, int TILE>
__device__ __forceinline__ void phase_a(const KParams& p, int64_t base, int tile_n, int16_t* s_list, int16_t* s_slot,
                                        uint8_t* s_flag, int* s_count_ptr) {
    const int tid = threadIdx.x;
    int& s_count = *s_count_ptr;
    if (p.mode == MODE_STEP && p.rep == PCGRL_REP_CELLULAR) cellular_rewrite<THREADS>(p, base, tile_n, s_flag);

    // ---------------- phase A: per-env action / reset, counters, change flag -----------------------
    for (int e = tid; e < TILE; e += THREADS) {
        bool need = false;
        if (e < tile_n) {
            const int64_t gid = base + e;
            if (p.mode == MODE_STEP) {
                const int cw = (p.rep == PCGRL_REP_CELLULAR) ? 3 * (int)s_flag[e] : apply_action(p, gid);
                need = step_counters(p, gid, cw);
            } else if (p.mode == MODE_RESET) {
                need = p.mask == nullptr || p.mask[gid] != 0;
                if (need) reset_env(p, gid);
            } else {
                need = true;
            }
        }
        // warp-aggregated append to the compact work list
        const unsigned bal = __ballot_sync(0xffffffffu, need);
        if (bal) {
            const int lane = tid & 31;
            int off = 0;
            if (lane == 0) off = atomicAdd(&s_count, __popc(bal));
            off = __shfl_sync(0xffffffffu, off, 0);
            if (need) {
                const int slot = off + __popc(bal & ((1u << lane) - 1u));
                s_list[slot] = (int16_t)e;
                s_slot[e] = (int16_t)slot;
            }
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// phase D (whole CTA, thread-per-env): reward = loss(new stats) - loss(old stats) in fp64, write stats.
//   s_stats[slot * K + k] holds the freshly computed stats of the listed envs.
// ------------------------------------------------------------------------------------------------
template <int THREADS, int K>
__device__ __forceinline__ void phase_d(const KParams& p, int64_t base, int tile_n, const int16_t* s_slot,
                                        const int32_t* s_stats) {
    const int tid = threadIdx.x;
    for (int e = tid; e < tile_n; e += THREADS) {
        const int slot = s_slot[e];
        if (slot < 0) continue;
        const int64_t gid = base + e;
        int32_t nw[K];
#pragma unroll
        for (int k = 0; k < K; ++k) nw[k] = s_stats[slot * K + k];
        if (p.mode == MODE_STATS) {
#pragma unroll
            for (int k = 0; k < K; ++k) p.stats_out[gid * K + k] = nw[k];
            continue;
        }
        finish_env<K>(p, gid, nw);
    }
}

}  // namespace pcgrl
