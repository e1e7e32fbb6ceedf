// Bit-board problem policies and per-thread stats state machines (binary, binary_holey, zelda), shared by the fused
// step kernel (step_bitboard.cu) and the split step kernels (step_split.cu).
#pragma once
#include "pcgrl_device.cuh"

namespace pcgrl {

// ------------------------------------------------------------------------------------------------
// Problem policies: planes (tile-code sets packed to bit-boards) + the per-thread stats state machine.
// Each machine is a flat loop: one board expansion per trip, with rare transitions -- so the 32 grids
// that share a warp execute the same instruction stream whatever phase each of them is in.
// ------------------------------------------------------------------------------------------------
struct BinaryProb {
    static constexpr int P = 1;
    static constexpr int K = 2;  // regions, path-length
    __host__ __device__ static constexpr uint32_t plane_mask(int p) { return 0x1u; }  // {empty}
};

struct ZeldaProb {
    static constexpr int P = 5;
    static constexpr int K = 7;  // player key door enemies regions nearest-enemy path-length
    // tiles: empty 0, solid 1, player 2, key 3, door 4, bat 5, scorpion 6, spider 7 (zelda_prob.py:20)
    __host__ __device__ static constexpr uint32_t plane_mask(int p) {
        return p == 0 ? 0xEDu   /* walkable {0,2,3,5,6,7}  zelda_ctrl_prob.py:101-104 */
             : p == 1 ? 0x04u   /* player */
             : p == 2 ? 0x08u   /* key */
             : p == 3 ? 0x10u   /* door */
             :          0xE0u;  /* enemies {5,6,7} */
    }
};

struct BinaryHoleyProb {
    static constexpr int P = 2;  // plane 0 {empty}; plane 1 holds no tile: the machine keeps the exit cell there
    static constexpr int K = 3;  // regions, path-length, connected-path-length
    __host__ __device__ static constexpr uint32_t plane_mask(int p) { return p == 0 ? 0x1u : 0x0u; }
};

// binary: regions + double-sweep longest path over the {empty} plane.
//   helper.calc_longest_path runs, per component, BFS(first tile) -> far tile -> BFS(far) and keeps the max.
//   Exact restatement used here: (1) isolated cells are components with eccentricity 0: count them with a
//   popcount; (2) for the other components run the first sweep one component at a time (start = lowest
//   remaining cell, far = lowest cell of the last non-empty level == np.argmax); (3) the second sweeps of
//   all components run at once as a single multi-source BFS from the set of far tiles -- components are
//   disconnected, so the number of levels until the joint frontier dies is max_c ecc(far_c).
template <int NW, bool TWO>
struct BinaryMachine {
    using Prob = BinaryProb;
    using B = Board<NW, TWO>;
    static constexpr bool HAS_CACHE = true;
    uint32_t avail[NW], front[NW], fars[NW];
    uint32_t* base;  // shared-memory copy of the passable cells (re-read for the joint sweep and the cache)
    int phase, level, ncomp;

    // Per-env search cache for the incremental machine (BinaryIncMachine, step_split.cu), written after the final
    // transition: [NW] passable board | [NW] far tiles (one per non-isolated component) | bit position of a cell
    // of a component that attains path-length (-1: none) | pad to 16 bytes.
    static constexpr int CACHE_BYTES = (2 * NW + 4) * 4;
    __device__ __forceinline__ void store_cache(uint32_t* c) const {
        int pos = -1;
#pragma unroll
        for (int i = NW - 1; i >= 0; --i)
            if (front[i]) pos = i * 32 + __ffs(front[i]) - 1;   // the last non-empty frontier of the joint sweep
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            c[i] = base[i];
            c[NW + i] = fars[i];
        }
        c[2 * NW] = (uint32_t)pos;
    }

    __device__ __forceinline__ void init(uint32_t* bb /* [P][NW] in shared memory */, const KParams&, int64_t) {
        uint32_t pass[NW], ones[NW], nb[NW];
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            pass[i] = bb[i];
            ones[i] = 0xFFFFFFFFu;
        }
        B::expand_and(pass, ones, nb);
        ncomp = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            const uint32_t iso = pass[i] & ~nb[i];
            ncomp += __popc(iso);
            avail[i] = pass[i] & ~iso;
            front[i] = 0;   // isolated cells stay in bb: the joint sweep can never reach them
            fars[i] = 0;
        }
        base = bb;
        phase = 0;
        level = 0;
    }
    // one board expansion; returns false (and changes nothing) when the frontier has died
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
    // the frontier died: next component / next phase; returns true when out[] holds the K stats
    __device__ __forceinline__ bool transition(int* out) {
        if (phase == 0) {
            uint32_t t[NW];
            B::minus_one(front, t);           // far tile of the component just swept (nothing on entry)
#pragma unroll
            for (int i = 0; i < NW; ++i) fars[i] |= front[i] & ~t[i];
            if (B::minus_one(avail, t)) {     // first tile of the next component
#pragma unroll
                for (int i = 0; i < NW; ++i) {
                    front[i] = avail[i] & ~t[i];
                    avail[i] &= t[i];
                }
                ++ncomp;
                return false;
            }
            phase = 1;  // joint second sweep from every far tile
            uint32_t any = 0;
#pragma unroll
            for (int i = 0; i < NW; ++i) {
                front[i] = fars[i];
                avail[i] = base[i] & ~fars[i];
                any |= fars[i];
            }
            level = 0;
            if (any) return false;
        }
        out[0] = ncomp;
        out[1] = level;
        return true;
    }
};

// binary_holey (envs/probs/binary/binary_holey_prob.py:59-93): the stats are taken on the BORDERED map
// (pcgrl_holey_env.py:52-53) whose border is solid except for the entrance and the exit.  The board built by
// phase B holds the level (one row per word); init() moves it one cell down-right into the border frame and
// digs the two holes.  regions = flood fill over the bordered board; then ONE BFS from the entrance:
// path-length = its last level (np.max of the dijkstra map), connected-path-length = the level that reaches
// the exit (0 when it never does: the reference maps -1 to 0, :69-77).
template <int NW, bool TWO>
struct BinaryHoleyMachine {
    static_assert(!TWO, "the bordered board keeps one row per word");
    static constexpr bool HAS_CACHE = false;
    using Prob = BinaryHoleyProb;
    using B = Board<NW, TWO>;
    uint32_t avail[NW], front[NW];
    uint32_t* bb;   // plane 0: bordered passable board, plane 1: the exit cell
    int phase, level, regions, connected, ey, ex;

    __device__ __forceinline__ void init(uint32_t* planes, const KParams& p, int64_t env) {
        bb = planes;
        const int32_t* h = p.holes + env * 4;
        ey = h[0];
        ex = h[1];
        const int xy = h[2], xx = h[3];
        uint32_t pass[NW], ones[NW], nb[NW];
#pragma unroll
        for (int i = 0; i < NW; ++i) pass[i] = i > 0 ? planes[i - 1] << 1 : 0u;
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            uint32_t xm = 0;
            if (i == xy && (unsigned)xx < 32u) xm = 1u << xx;
            if (i == ey && (unsigned)ex < 32u) pass[i] |= 1u << ex;
            pass[i] |= xm;
            planes[i] = pass[i];
            planes[NW + i] = xm;
            ones[i] = 0xFFFFFFFFu;
        }
        B::expand_and(pass, ones, nb);
        regions = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            const uint32_t iso = pass[i] & ~nb[i];
            regions += __popc(iso);
            avail[i] = pass[i] & ~iso;
            front[i] = 0;
        }
        phase = 0;
        level = 0;
        connected = 0;
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
        if (phase == 1) {
            uint32_t hit = 0;
#pragma unroll
            for (int i = 0; i < NW; ++i) hit |= n[i] & bb[NW + i];
            if (hit) connected = level;
        }
        return true;
    }
    __device__ __forceinline__ bool transition(int* out) {
        if (phase == 0) {
            uint32_t t[NW];
            if (B::minus_one(avail, t)) {
#pragma unroll
                for (int i = 0; i < NW; ++i) {
                    front[i] = avail[i] & ~t[i];
                    avail[i] &= t[i];
                }
                ++regions;
                return false;
            }
            phase = 1;   // BFS from the entrance over the whole bordered board
            level = 0;
#pragma unroll
            for (int i = 0; i < NW; ++i) {
                front[i] = (i == ey && (unsigned)ex < 32u) ? 1u << ex : 0u;
                avail[i] = bb[i] & ~front[i];
            }
            return false;
        }
        out[0] = regions;
        out[1] = level;
        out[2] = connected;
        return true;
    }
};

// zelda: tile counts, regions over the walkable plane, then (player == 1) BFS from the player:
// nearest-enemy = first level >= 1 that touches an enemy, d(player->key) = level that touches the key;
// then (key == 1 && door == 1) BFS from the key over walkable+door: d(key->door).  Unreached = -1 each
// (run_dijkstra's fill value), added raw (zelda_ctrl_prob.py:134-150).
template <int NW, bool TWO>
struct ZeldaMachine {
    static constexpr bool HAS_CACHE = false;
    using Prob = ZeldaProb;
    using B = Board<NW, TWO>;
    uint32_t avail[NW], front[NW];
    const uint32_t* bb;  // planes in shared memory: walk, player, key, door, enemy
    int phase, level, regions, near, dkey, ddoor;
    int n_player, n_key, n_door, n_enemy;

    __device__ __forceinline__ void load(int plane, uint32_t (&x)[NW]) const {
#pragma unroll
        for (int i = 0; i < NW; ++i) x[i] = bb[plane * NW + i];
    }
    __device__ __forceinline__ void init(uint32_t* planes, const KParams&, int64_t) {
        bb = planes;
        uint32_t walk[NW], t[NW], ones[NW], nb[NW];
        load(0, walk);
        load(1, t);
        n_player = B::popcount(t);
        load(2, t);
        n_key = B::popcount(t);
        load(3, t);
        n_door = B::popcount(t);
        load(4, t);
        n_enemy = B::popcount(t);
#pragma unroll
        for (int i = 0; i < NW; ++i) ones[i] = 0xFFFFFFFFu;
        B::expand_and(walk, ones, nb);
        regions = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            const uint32_t iso = walk[i] & ~nb[i];
            regions += __popc(iso);
            avail[i] = walk[i] & ~iso;
            front[i] = 0;
        }
        phase = 0;
        level = 0;
        near = 0;
        dkey = -1;
        ddoor = -1;
    }
    __device__ __forceinline__ bool expand() {
        uint32_t n[NW];
        if (!B::expand_and(front, avail, n)) return false;
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            avail[i] ^= n[i];
            front[i] = n[i];
        }
        ++level;
        if (phase == 1) {
            uint32_t t[NW];
            load(4, t);
            if (near == 0 && B::any_and(n, t)) near = level;
            load(2, t);
            if (B::any_and(n, t)) dkey = level;
        } else if (phase == 2) {
            uint32_t t[NW];
            load(3, t);
            if (B::any_and(n, t)) ddoor = level;
        }
        return true;
    }
    __device__ __forceinline__ bool transition(int* out) {
        if (phase == 0) {  // region flood fill, one component at a time
            uint32_t t[NW];
            if (B::minus_one(avail, t)) {
#pragma unroll
                for (int i = 0; i < NW; ++i) {
                    front[i] = avail[i] & ~t[i];
                    avail[i] &= t[i];
                }
                ++regions;
                return false;
            }
            if (n_player == 1 && (n_enemy > 0 || (n_key == 1 && n_door == 1))) {
                phase = 1;  // BFS from the player over the walkable plane
                uint32_t walk[NW];
                load(0, walk);
                load(1, front);
#pragma unroll
                for (int i = 0; i < NW; ++i) avail[i] = walk[i] & ~front[i];
                level = 0;
                return false;
            }
            phase = 3;
        } else if (phase == 1) {
            if (n_key == 1 && n_door == 1) {
                phase = 2;  // BFS from the key over walkable + door
                uint32_t walk[NW], door[NW];
                load(0, walk);
                load(3, door);
                load(2, front);
#pragma unroll
                for (int i = 0; i < NW; ++i) avail[i] = (walk[i] | door[i]) & ~front[i];
                level = 0;
                return false;
            }
            phase = 3;
        }
        out[0] = n_player;
        out[1] = n_key;
        out[2] = n_door;
        out[3] = n_enemy;
        out[4] = regions;
        out[5] = near;
        out[6] = (n_player == 1 && n_key == 1 && n_door == 1) ? dkey + ddoor : 0;
        return true;
    }
};

// ------------------------------------------------------------------------------------------------
// 16 tile codes (one 128-bit load) -> one 16-bit membership mask per plane (bit i = cell i in the plane).
// Tile codes are < 8 for every bit-board problem, so a plane is an 8-entry 0/1 table that PRMT looks up
// for 4 cells at once; the multiply then gathers the four 0/1 bytes into bits 24..27.
// ------------------------------------------------------------------------------------------------
__host__ __device__ constexpr uint32_t lut_bytes(uint32_t mask, int first) {
    return ((mask >> first) & 1u) | (((mask >> (first + 1)) & 1u) << 8) | (((mask >> (first + 2)) & 1u) << 16) |
           (((mask >> (first + 3)) & 1u) << 24);
}
template <class Prob>
__device__ __forceinline__ void pack16(const uint4 v, uint32_t (&out)[Prob::P]) {
    const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < Prob::P; ++q) out[q] = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t t = w4[k] | (w4[k] >> 4);
        const uint32_t sel = ((t & 0xFFu) | ((t >> 8) & 0xFF00u)) & 0x7777u;  // 4 nibbles = 4 tile codes
#pragma unroll
        for (int q = 0; q < Prob::P; ++q) {
            const uint32_t b = __byte_perm(lut_bytes(Prob::plane_mask(q), 0), lut_bytes(Prob::plane_mask(q), 4), sel);
            out[q] |= ((b * 0x01020408u) >> 24) << (4 * k);
        }
    }
}

// barrier of the threads that cooperate in stage_boards: a warp (GROUP == 32) or the whole CTA
template <int GROUP>
__device__ __forceinline__ void group_sync() {
    if constexpr (GROUP == 32) __syncwarp();
    else __syncthreads();
}

// Coalesced 128-bit loads of n level grids -> per-plane bit-boards in shared memory, P * NW words per slot (plane q of
// slot i at bb[i * P * NW + q * NW]).  The GROUP threads that cooperate call it together, rank = the thread's index
// among them; row(i) is the grid of slot i.  On return the boards are complete for the whole group.
template <class Prob, int NW, bool TWO, int GROUP, class Row>
__device__ __forceinline__ void stage_boards(const KParams& p, int rank, int n, uint32_t* bb, Row row) {
    constexpr int P = Prob::P;
    constexpr int BBW = P * NW;
    const int chunks = p.row_stride / 16;
    const int W = p.d1;
    const bool word_is_32_bytes = TWO ? (W == 16) : (W == 32);
    if (word_is_32_bytes) {
        // a board word is exactly 32 consecutive cells: one thread builds one word, no atomics
        for (int i = rank; i < n * NW; i += GROUP) {
            const int slot = i / NW, j = i - slot * NW;
            const int8_t* g = row(slot) + j * 32;
            uint32_t lo[P], hi[P];
#pragma unroll
            for (int q = 0; q < P; ++q) lo[q] = hi[q] = 0;
            if (2 * j < chunks) pack16<Prob>(*(const uint4*)g, lo);
            if (2 * j + 1 < chunks) pack16<Prob>(*(const uint4*)(g + 16), hi);
#pragma unroll
            for (int q = 0; q < P; ++q) bb[slot * BBW + q * NW + j] = lo[q] | (hi[q] << 16);
        }
    } else {
        for (int i = rank; i < n * BBW; i += GROUP) bb[i] = 0;
        group_sync<GROUP>();
        for (int i = rank; i < n * chunks; i += GROUP) {
            const int slot = i / chunks, c = i - slot * chunks;
            uint32_t lin[P];
            pack16<Prob>(*(const uint4*)(row(slot) + c * 16), lin);
            uint32_t* sb = bb + slot * BBW;
            int cell = c * 16;
            const int end = min(cell + 16, p.cells);
            int y = cell / W, x = cell - y * W;
            while (cell < end) {   // one row segment at a time (at most ceil(16/W)+1 of them)
                const int len = min(W - x, end - cell);
                const int word = TWO ? (y >> 1) : y;
                const int sh = TWO ? ((y & 1) * 16 + x) : x;
                const uint32_t m = (1u << len) - 1u;
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    const uint32_t seg = (lin[q] >> (cell - c * 16)) & m;
                    if (seg) atomicOr(&sb[q * NW + word], seg << sh);
                }
                cell += len;
                x = 0;
                ++y;
            }
        }
    }
    group_sync<GROUP>();
}

}  // namespace pcgrl
