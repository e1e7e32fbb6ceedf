// sokoban: fused env step with warp-per-grid get_stats, including the reference's solver.
//
// Reference path replaced (paths relative to /root/reference/control_pcgrl/envs/probs/sokoban/):
//   sokoban_prob.py:160-180 + sokoban_ctrl_prob.py:58-65   get_stats (counts, regions, dist-win, sol-length, ratio)
//   sokoban_prob.py:99-148                                  _run_game: BFS -> A*(1) -> A*(0.5) -> A*(0), 10 000 iterations each
//   sokoban/engine.py:56-74 BFSAgent, :96-119 AStarAgent, :121-363 State (update, deadlocks, heuristic, key)
//
// State = player position + crate positions in list order (the reference's visited key lists the crates in
// order, engine.py:329-335), one byte each (position = y * BW + x in the '#'-framed level), packed in a uint4.
// A node = state + depth + heuristic; parents are not kept (only len(solution) = depth is observable).
// Node pools, the A* heap and the visited hash table live in a per-warp slice of the global scratch; the
// level itself (solid / deadlock bit masks, target list) lives in shared memory.
//
// Exactness notes (SURVEY.md A-16, A-18):
//   * iterations count every pop, also of already visited keys; win is tested on pop, before the visited test;
//   * a state wins iff its heuristic is 0 (#crates == #targets > 0 is a precondition of running the solver and
//     the greedy crate->target matching is then a perfect matching at distance 0), so the stored heuristic
//     doubles as the win flag;
//   * queue.PriorityQueue == heapq on Node.__lt__ = h + balance * depth: the binary heap below performs CPython's
//     heappush / heappop moves (_siftdown / _siftup) with `<` only; keys are the exact integers 2h + (2 balance) d;
//   * if the BFS empties its queue without a win, each A* would pop exactly the same multiset of nodes
//     (1 + sum of children over all reachable states) and end with best heuristic = min over reachable states,
//     so dist-win is taken from the BFS directly; the A* passes only run when the BFS hit the iteration cap.
#include "step_search.cuh"

namespace pcgrl {

constexpr int SOK_POWER = 10000;                 // sokoban_prob.py:40 _solver_power
constexpr int SOK_NODES = 4 * SOK_POWER + 8;     // root + <= 4 children per iteration
constexpr int SOK_TABLE = 32768;                 // visited hash slots (<= 10 000 insertions per search)
constexpr int SOK_MAX_CRATES = 15;
constexpr int SOK_MAX_CTAS_PER_SM = 2;   // A/B on B200: 2 / 3 / 4 CTAs per SM change nothing (bounded by the longest solve)
constexpr int SOK_MAX_CTAS = 160 * SOK_MAX_CTAS_PER_SM;   // sizes the global scratch (>= 148 SMs x CTAs per SM)

struct SokScratch {
    // byte offsets inside one warp's slice
    static constexpr size_t header = 0;                                    // u32 generation counter (+pad)
    static constexpr size_t state = 16;                                    // uint4[SOK_NODES]
    static constexpr size_t meta = state + sizeof(uint4) * SOK_NODES;      // u32[SOK_NODES]: depth | h << 16
    static constexpr size_t heap = meta + 4 * (size_t)SOK_NODES;           // u32[SOK_NODES]: idx | key << 16
    static constexpr size_t table = heap + 4 * (size_t)SOK_NODES;          // u32[SOK_TABLE]: idx | gen << 16
    static constexpr size_t total = (table + 4 * (size_t)SOK_TABLE + 255) / 256 * 256;
};

// Deferred solver jobs (the front of the global scratch, before the per-warp slices).  get_stats itself is cheap
// for almost every level (counts + regions); 1.3 % of random 5x5 levels meet the solver preconditions, their BFS
// takes 53 pops on average, and 1 in 4 000 of those hits the 10 000-pop cap and then runs the three A* passes
// (10 000 dependent heap operations each).  Solving inline, one such level used to hold its warp, its CTA and
// then the whole launch for ~85 ms while 94 % of the GPU idled.  So the step kernel only RECORDS the levels that
// need the solver (k_step_search, pass 1); k_sokoban_solve runs their BFS with 32 pops per round on a persistent
// grid of warps pulling jobs from a global counter; levels whose BFS hit the cap become three independent A* jobs
// for k_sokoban_astar (one single-warp CTA each, heap and visited table in 224 KB of shared memory);
// k_sokoban_combine picks the result in the reference's order and re-arms the lists.
struct SokJobs {
    static constexpr int CAP = 1 << 20;          // jobs per launch; beyond it levels are solved inline (pass 1)
    static constexpr int ASTAR_CAP = 4096;       // levels per launch whose A* passes run as separate jobs
    static constexpr size_t header = 0;          // u32: [0] n_jobs, [1] next job, [2] n_astar, [3] next A* job
    static constexpr size_t jobs = 256;          // int32[CAP][8]: env (or grid index), old stats [7]
    static constexpr size_t astar = jobs + (size_t)CAP * 32;               // int32[ASTAR_CAP]: job index
    static constexpr size_t results = astar + (size_t)ASTAR_CAP * 4;       // int32[ASTAR_CAP][3][4]: won, depth, best h
    static constexpr size_t total = (results + (size_t)ASTAR_CAP * 48 + 255) / 256 * 256;
};

int64_t sokoban_scratch_bytes() { return (int64_t)SokJobs::total + (int64_t)SokScratch::total * SOK_MAX_CTAS * SEARCH_WARPS; }

struct SokobanProb {
    static constexpr int K = 7;   // player crate target regions dist-win sol-length ratio

    struct Ctx {
        int H, W, BW, BH;
        // shared memory
        uint8_t* stage;      // raw grid bytes
        uint32_t* solid;     // [8] bit p = '#'
        uint32_t* dead;      // [8] bit p = static deadlock cell
        uint8_t* tpos;       // [16] target positions in scan order
        uint8_t* cpos;       // [256] scratch list (crates, then corners)
        uint16_t* rows;      // [16] passable rows, then [256] union-find parents
        // global scratch slice
        uint32_t* hdr;
        uint4* state;
        uint32_t *meta, *heap, *table;
        int nt;              // #targets == #crates while solving
        uint32_t magic_bw;
    };

    __host__ __device__ static int smem_bytes(int row_stride) {
        return (row_stride + 15) / 16 * 16 + 32 + 32 + 16 + 256 + 2 * (16 + 256);
    }

    __device__ static Ctx make_ctx(const KParams& p, uint8_t* ws, int global_warp) {
        Ctx c;
        c.H = p.d0; c.W = p.d1;
        c.BW = c.W + 2; c.BH = c.H + 2;
        int o = 0;
        c.stage = ws + o;             o += (p.row_stride + 15) / 16 * 16;
        c.solid = (uint32_t*)(ws + o); o += 32;
        c.dead = (uint32_t*)(ws + o);  o += 32;
        c.tpos = ws + o;              o += 16;
        c.cpos = ws + o;              o += 256;
        c.rows = (uint16_t*)(ws + o);
        uint8_t* g = (uint8_t*)p.scratch + SokJobs::total + (size_t)global_warp * SokScratch::total;
        c.hdr = (uint32_t*)(g + SokScratch::header);
        c.state = (uint4*)(g + SokScratch::state);
        c.meta = (uint32_t*)(g + SokScratch::meta);
        c.heap = (uint32_t*)(g + SokScratch::heap);
        c.table = (uint32_t*)(g + SokScratch::table);
        c.nt = 0;
        c.magic_bw = div_magic(c.BW);
        return c;
    }

    // ---- state helpers (registers) -------------------------------------------------------------------------
    __device__ static __forceinline__ uint32_t get_byte(const uint4& s, int i) {
        const uint32_t w = i < 4 ? s.x : (i < 8 ? s.y : (i < 12 ? s.z : s.w));
        return (w >> ((i & 3) * 8)) & 0xFFu;
    }
    __device__ static __forceinline__ void set_byte(uint4& s, int i, uint32_t v) {
        const uint32_t sh = (i & 3) * 8, m = ~(0xFFu << sh), b = v << sh;
        if (i < 4) s.x = (s.x & m) | b;
        else if (i < 8) s.y = (s.y & m) | b;
        else if (i < 12) s.z = (s.z & m) | b;
        else s.w = (s.w & m) | b;
    }
    // index (1..15) of the state byte holding crate position `pos`, or 0 (engine.py:257-261 checkCrateLocation)
    __device__ static __forceinline__ int crate_byte(const uint4& s, uint32_t pos) {
        const uint32_t pat = pos * 0x01010101u;
        uint32_t m = __vcmpeq4(s.x, pat) & 0xFFFFFF00u;    // byte 0 is the player
        if (m) return (__ffs(m) - 1) >> 3;
        m = __vcmpeq4(s.y, pat);
        if (m) return 4 + ((__ffs(m) - 1) >> 3);
        m = __vcmpeq4(s.z, pat);
        if (m) return 8 + ((__ffs(m) - 1) >> 3);
        m = __vcmpeq4(s.w, pat);
        if (m) return 12 + ((__ffs(m) - 1) >> 3);
        return 0;
    }
    __device__ static __forceinline__ bool bit(const uint32_t* m, uint32_t p) { return (m[p >> 5] >> (p & 31)) & 1u; }

    // engine.py:279-293 getHeuristic: greedy crate -> nearest remaining target (first minimum, strict '>')
    __device__ static int heuristic(const Ctx& c, const uint4& s) {
        uint32_t remaining = (1u << c.nt) - 1u;
        int total = 0;
        for (int i = 0; i < c.nt; ++i) {
            const int cp = get_byte(s, 1 + i), cy = div_by(cp, c.magic_bw), cx = cp - cy * c.BW;
            int best = c.BW + c.BH, bi = -1, bd = 0;
            for (uint32_t r = remaining; r; r &= r - 1) {
                const int j = __ffs(r) - 1;
                const int tp = c.tpos[j], ty = div_by(tp, c.magic_bw);
                const int d = abs(cx - (tp - ty * c.BW)) + abs(cy - ty);
                if (bi < 0) {          // bestMatch defaults to the first remaining target
                    bi = j;
                    bd = d;
                }
                if (best > d) {
                    best = d;
                    bi = j;
                    bd = d;
                }
            }
            total += bd;
            remaining &= ~(1u << bi);
        }
        return total;
    }

    __device__ static __forceinline__ uint32_t hash_state(const uint4& s) {
        uint32_t h = s.x * 0x9E3779B1u;
        h = (h ^ (h >> 15)) + s.y * 0x85EBCA77u;
        h = (h ^ (h >> 13)) + s.z * 0xC2B2AE3Du;
        h = (h ^ (h >> 16)) + s.w * 0x27D4EB2Fu;
        h ^= h >> 15;
        h *= 0x2C1B3C6Du;
        h ^= h >> 12;
        return h;
    }

    // visited set (lane 0 only): true if `s` was already there, else inserts node `idx`
    __device__ static bool visited_test_and_set(const Ctx& c, const uint4& s, int idx, uint32_t gen) {
        uint32_t i = hash_state(s) & (SOK_TABLE - 1);
        for (;;) {
            const uint32_t slot = c.table[i];
            if ((slot >> 16) != gen) {
                c.table[i] = (uint32_t)idx | (gen << 16);
                return false;
            }
            const uint4 o = c.state[slot & 0xFFFFu];
            if (o.x == s.x && o.y == s.y && o.z == s.z && o.w == s.w) return true;
            i = (i + 1) & (SOK_TABLE - 1);
        }
    }

    // ---- CPython heapq on (key, idx) entries, lane 0 only --------------------------------------------------
    __device__ static __forceinline__ void sift_down(uint32_t* heap, int start, int pos) {
        const uint32_t item = heap[pos];
        while (pos > start) {
            const int parent = (pos - 1) >> 1;
            const uint32_t pe = heap[parent];
            if ((item >> 16) < (pe >> 16)) {
                heap[pos] = pe;
                pos = parent;
                continue;
            }
            break;
        }
        heap[pos] = item;
    }
    __device__ static __forceinline__ void heap_push(uint32_t* heap, int& n, uint32_t entry) {
        heap[n] = entry;
        sift_down(heap, 0, n);
        ++n;
    }
    __device__ static __forceinline__ uint32_t heap_pop(uint32_t* heap, int& n) {
        const uint32_t last = heap[--n];
        if (n == 0) return last;
        const uint32_t ret = heap[0];
        int pos = 0, child = 1;
        while (child < n) {
            const int right = child + 1;
            uint32_t ce = heap[child];
            if (right < n) {
                const uint32_t re = heap[right];
                if (!((ce >> 16) < (re >> 16))) {
                    child = right;
                    ce = re;
                }
            }
            heap[pos] = ce;
            pos = child;
            child = 2 * pos + 1;
        }
        heap[pos] = last;
        sift_down(heap, 0, pos);
        return ret;
    }

    // ---- one search: mode 0 = BFSAgent, 1..3 = AStarAgent with 2*balance = 2, 1, 0 ---------------------------
    // Returns true on win (depth in `out_depth`); else best heuristic in `out_h`; `exhausted` = queue ran empty.
    __device__ static bool search(Ctx& c, const uint4 root, int root_h, int mode, int lane, int& out_depth, int& out_h,
                                  bool& exhausted) {
        const int bal2 = mode == 1 ? 2 : (mode == 2 ? 1 : 0);
        // new generation of the visited table (cleared only when the 16-bit tag wraps)
        uint32_t gen = 0;
        if (lane == 0) gen = *c.hdr + 1;
        gen = __shfl_sync(0xffffffffu, gen, 0);
        if (gen > 0xFFFFu) {
            for (int i = lane; i < SOK_TABLE; i += 32) c.table[i] = 0;
            gen = 1;
        }
        if (lane == 0) {
            *c.hdr = gen;
            c.state[0] = root;
            c.meta[0] = (uint32_t)root_h << 16;
            c.heap[0] = (uint32_t)(2 * root_h) << 16;
        }
        __syncwarp();
        int n_nodes = 1, head = 0, hn = 1;
        int best_h = 0x7FFFFFFF, best_d = 0, iters = 0;
        const int delta = lane == 0 ? -1 : (lane == 1 ? 1 : (lane == 2 ? -c.BW : c.BW));   // engine.py:3 L R U D
        for (;;) {
            const bool empty = mode == 0 ? head >= n_nodes : hn == 0;
            if (iters >= SOK_POWER || empty) {
                exhausted = empty;
                break;
            }
            ++iters;
            // pop + visited test on lane 0, broadcast
            int cur = 0, seen = 0;
            if (lane == 0) {
                cur = mode == 0 ? head : (int)(heap_pop(c.heap, hn) & 0xFFFFu);
            }
            cur = __shfl_sync(0xffffffffu, cur, 0);
            if (mode == 0) ++head;
            const uint4 s = c.state[cur];
            const uint32_t m = c.meta[cur];
            const int h = m >> 16, d = m & 0xFFFFu;
            if (h == 0) {                                     // checkWin (engine.py:64 / :108)
                out_depth = d;
                return true;
            }
            if (lane == 0) seen = visited_test_and_set(c, s, cur, gen);
            seen = __shfl_sync(0xffffffffu, seen, 0);
            if (mode != 0) hn = __shfl_sync(0xffffffffu, hn, 0);
            if (seen) continue;
            if (h < best_h || (h == best_h && d < best_d)) {  // engine.py:66-70
                best_h = h;
                best_d = d;
            }
            // children (Node.getChildren, engine.py:14-24): lane = direction
            bool valid = false;
            uint4 cs = s;
            int ch = 0;
            if (lane < 4) {
                const uint32_t pp = s.x & 0xFFu, np = pp + delta;
                if (!bit(c.solid, np)) {
                    const int cb = crate_byte(s, np);
                    if (cb == 0) {                            // plain move
                        cs.x = (s.x & 0xFFFFFF00u) | np;
                        valid = true;
                        ch = h;
                    } else {                                  // push crate `cb - 1`
                        const uint32_t cp = np + delta;
                        if (!bit(c.solid, cp) && crate_byte(s, cp) == 0) {
                            set_byte(cs, cb, cp);
                            cs.x = (cs.x & 0xFFFFFF00u) | np;
                            bool deadlocked = false;          // checkDeadlock: any crate on a deadlock cell
                            for (int i = 0; i < c.nt; ++i) deadlocked |= bit(c.dead, get_byte(cs, 1 + i));
                            if (!deadlocked) {
                                valid = true;
                                ch = heuristic(c, cs);
                            }
                        }
                    }
                }
            }
            const unsigned vm = __ballot_sync(0xffffffffu, valid);
            if (valid) {
                const int idx = n_nodes + __popc(vm & ((1u << lane) - 1u));
                c.state[idx] = cs;
                c.meta[idx] = ((uint32_t)ch << 16) | (uint32_t)(d + 1);
            }
            const int nc = __popc(vm);
            if (mode != 0) {
                __syncwarp();
                if (lane == 0) {
                    for (int k = 0; k < nc; ++k) {
                        const int idx = n_nodes + k;
                        const uint32_t mm = c.meta[idx];
                        const uint32_t key = 2u * (mm >> 16) + (uint32_t)bal2 * (mm & 0xFFFFu);
                        heap_push(c.heap, hn, (uint32_t)idx | (key << 16));
                    }
                }
                hn = __shfl_sync(0xffffffffu, hn, 0);
            }
            n_nodes += nc;
            __syncwarp();
        }
        out_h = best_h;
        return false;
    }

    // ---- lane-parallel BFSAgent (engine.py:56-74): 32 queue entries per round ---------------------------------
    // The FIFO order only matters through (a) the pop count (every pop counts, also of visited keys), (b) which of
    // several equal states is expanded (the first one popped) and (c) the order in which children are appended.
    // A round takes the next B <= 32 entries (never past the iteration cap), tests the win in queue order, drops
    // entries whose state was expanded in an earlier round (table probe) or by a LOWER lane of this round
    // (__match_any on the state hash, verified on the full state), inserts the survivors, and appends their
    // children lane by lane, direction by direction -- exactly the queue the sequential loop builds.
    __device__ static bool table_contains(const Ctx& c, const uint4& s, uint32_t hash, uint32_t gen) {
        uint32_t i = hash & (SOK_TABLE - 1);
        for (;;) {
            const uint32_t slot = c.table[i];
            if ((slot >> 16) != gen) return false;
            const uint4 o = c.state[slot & 0xFFFFu];
            if (o.x == s.x && o.y == s.y && o.z == s.z && o.w == s.w) return true;
            i = (i + 1) & (SOK_TABLE - 1);
        }
    }
    __device__ static void table_insert(const Ctx& c, uint32_t hash, int idx, uint32_t gen) {
        uint32_t i = hash & (SOK_TABLE - 1);
        const uint32_t val = (uint32_t)idx | (gen << 16);
        for (;;) {
            const uint32_t slot = c.table[i];
            if ((slot >> 16) != gen) {
                if (atomicCAS(&c.table[i], slot, val) == slot) return;
                continue;      // another lane of this round took the slot: look at it again
            }
            i = (i + 1) & (SOK_TABLE - 1);
        }
    }
    // one child of state s in direction `dir` (engine.py:14-24 getChildren, :295-327 update)
    __device__ static __forceinline__ bool make_child(const Ctx& c, const uint4& s, int h, int dir, uint4& cs, int& ch) {
        const int delta = dir == 0 ? -1 : (dir == 1 ? 1 : (dir == 2 ? -c.BW : c.BW));   // engine.py:3 L R U D
        const uint32_t pp = s.x & 0xFFu, np = pp + delta;
        if (bit(c.solid, np)) return false;
        cs = s;
        const int cb = crate_byte(s, np);
        if (cb == 0) {                            // plain move
            cs.x = (s.x & 0xFFFFFF00u) | np;
            ch = h;
            return true;
        }
        const uint32_t cp = np + delta;           // push crate `cb - 1`
        if (bit(c.solid, cp) || crate_byte(s, cp) != 0) return false;
        set_byte(cs, cb, cp);
        cs.x = (cs.x & 0xFFFFFF00u) | np;
        bool deadlocked = false;                  // checkDeadlock: any crate on a deadlock cell
        for (int i = 0; i < c.nt; ++i) deadlocked |= bit(c.dead, get_byte(cs, 1 + i));
        if (deadlocked) return false;
        ch = heuristic(c, cs);
        return true;
    }
    __device__ static bool bfs_parallel(Ctx& c, const uint4 root, int root_h, int lane, int& out_depth, int& out_h,
                                        bool& exhausted) {
        uint32_t gen = 0;
        if (lane == 0) gen = *c.hdr + 1;
        gen = __shfl_sync(0xffffffffu, gen, 0);
        if (gen > 0xFFFFu) {
            for (int i = lane; i < SOK_TABLE; i += 32) c.table[i] = 0;
            gen = 1;
        }
        if (lane == 0) {
            *c.hdr = gen;
            c.state[0] = root;
            c.meta[0] = (uint32_t)root_h << 16;
        }
        __syncwarp();
        int n_nodes = 1, head = 0, iters = 0;
        uint32_t best = 0xFFFFFFFFu;               // (h << 16 | depth) of the best expanded node (engine.py:66-70)
        for (;;) {
            const int avail = n_nodes - head;
            if (iters >= SOK_POWER || avail == 0) {
                exhausted = avail == 0;
                break;
            }
            const int B = min(min(32, avail), SOK_POWER - iters);
            const bool mine = lane < B;
            uint4 s = make_uint4(0, 0, 0, 0);
            uint32_t m = 0xFFFF0000u;
            if (mine) {
                s = c.state[head + lane];
                m = c.meta[head + lane];
            }
            const int h = m >> 16, d = m & 0xFFFFu;
            const unsigned wins = __ballot_sync(0xffffffffu, mine && h == 0);      // checkWin, in queue order
            if (wins) {
                out_depth = __shfl_sync(0xffffffffu, d, __ffs(wins) - 1);
                return true;
            }
            const uint32_t hash = hash_state(s);
            bool fresh = mine && !table_contains(c, s, hash, gen);
            // duplicates inside the round: the lowest lane holding a state expands it
            const unsigned mm = __ballot_sync(0xffffffffu, mine);
            bool dup = false;
            unsigned clash = 0;
            if (mine) {
                const unsigned grp = __match_any_sync(mm, hash);
                const int lead = __ffs(grp) - 1;
                const uint4 ls = make_uint4(__shfl_sync(mm, s.x, lead), __shfl_sync(mm, s.y, lead),
                                            __shfl_sync(mm, s.z, lead), __shfl_sync(mm, s.w, lead));
                const bool same = ls.x == s.x && ls.y == s.y && ls.z == s.z && ls.w == s.w;
                dup = lead != lane && same;
                clash = __ballot_sync(mm, lead != lane && !same);
            }
            clash = __shfl_sync(0xffffffffu, clash, 0);
            if (clash) {       // two different states share a 32-bit hash (practically never): compare all pairs
                dup = false;
                for (int j = 0; j < B; ++j) {
                    const uint4 o = make_uint4(__shfl_sync(0xffffffffu, s.x, j), __shfl_sync(0xffffffffu, s.y, j),
                                               __shfl_sync(0xffffffffu, s.z, j), __shfl_sync(0xffffffffu, s.w, j));
                    dup |= j < lane && o.x == s.x && o.y == s.y && o.z == s.z && o.w == s.w;
                }
            }
            fresh = fresh && !dup;
            __syncwarp();
            if (fresh) table_insert(c, hash, head + lane, gen);
            best = min(best, __reduce_min_sync(0xffffffffu, fresh ? (((uint32_t)h << 16) | (uint32_t)d) : 0xFFFFFFFFu));
            // children of the survivors, appended lane by lane, L R U D inside a lane
            uint4 cs[4];
            int chh[4];
            unsigned okm = 0;
            if (fresh) {
#pragma unroll
                for (int dir = 0; dir < 4; ++dir)
                    if (make_child(c, s, h, dir, cs[dir], chh[dir])) okm |= 1u << dir;
            }
            const int cnt = __popc(okm);
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            int at = n_nodes + incl - cnt;
#pragma unroll
            for (int dir = 0; dir < 4; ++dir)
                if (okm & (1u << dir)) {
                    c.state[at] = cs[dir];
                    c.meta[at] = ((uint32_t)chh[dir] << 16) | (uint32_t)(d + 1);
                    ++at;
                }
            n_nodes += total;
            head += B;
            iters += B;
            __syncwarp();
        }
        out_h = (int)(best >> 16);
        return false;
    }

    // ---- AStarAgent (engine.py:96-119) with the heap and the visited table in shared memory --------------------
    // Same pops, same order as search() modes 1..3; only where the data lives differs: the binary heap (<= 40 008
    // entries) and a 32 768-slot table of 16-bit node indices sit in the CTA's shared memory, so a pop is ~15
    // shared-memory round trips instead of ~15 trips to L2.
    static constexpr int ASTAR_TABLE = 32768;
    __device__ static bool astar_smem(Ctx& c, const uint4 root, int root_h, int mode, int lane, uint32_t* heap,
                                      uint16_t* table, int& out_depth, int& out_h) {
        const int bal2 = mode == 1 ? 2 : (mode == 2 ? 1 : 0);
        {
            uint4* t4 = (uint4*)table;
            for (int i = lane; i < ASTAR_TABLE * 2 / 16; i += 32) t4[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
        }
        if (lane == 0) {
            c.state[0] = root;
            c.meta[0] = (uint32_t)root_h << 16;
            heap[0] = (uint32_t)(2 * root_h) << 16;
        }
        __syncwarp();
        int n_nodes = 1, hn = 1;
        int best_h = 0x7FFFFFFF, best_d = 0, iters = 0;
        const int delta = lane == 0 ? -1 : (lane == 1 ? 1 : (lane == 2 ? -c.BW : c.BW));
        for (;;) {
            if (iters >= SOK_POWER || hn == 0) break;
            ++iters;
            int seen = 0;
            // the node about to be popped is the heap's root: its state (L2) is requested before lane 0 walks the heap
            // (~13 dependent shared-memory levels), so the two latencies overlap instead of adding up
            const int cur = (int)(heap[0] & 0xFFFFu);
            __syncwarp();                        // every lane has read the root before lane 0 rewrites the heap
            const uint4 s = c.state[cur];
            const uint32_t m = c.meta[cur];
            if (lane == 0) heap_pop(heap, hn);
            const int h = m >> 16, d = m & 0xFFFFu;
            if (h == 0) {
                out_depth = d;
                return true;
            }
            // (the table lookup on lane 1, as a second instruction stream next to lane 0's heap walk, gains nothing:
            // A* launch 8.84 against 8.69 ms)
            if (lane == 0) {
                uint32_t i = hash_state(s) & (ASTAR_TABLE - 1);
                for (;;) {
                    const uint32_t slot = table[i];
                    if (slot == 0xFFFFu) {
                        table[i] = (uint16_t)cur;
                        break;
                    }
                    const uint4 o = c.state[slot];
                    if (o.x == s.x && o.y == s.y && o.z == s.z && o.w == s.w) {
                        seen = 1;
                        break;
                    }
                    i = (i + 1) & (ASTAR_TABLE - 1);
                }
            }
            seen = __shfl_sync(0xffffffffu, seen, 0);
            hn = __shfl_sync(0xffffffffu, hn, 0);
            if (seen) continue;
            if (h < best_h || (h == best_h && d < best_d)) {
                best_h = h;
                best_d = d;
            }
            bool valid = false;
            uint4 cs = s;
            int ch = 0;
            if (lane < 4) {
                const uint32_t pp = s.x & 0xFFu, np = pp + delta;
                if (!bit(c.solid, np)) {
                    const int cb = crate_byte(s, np);
                    if (cb == 0) {
                        cs.x = (s.x & 0xFFFFFF00u) | np;
                        valid = true;
                        ch = h;
                    } else {
                        const uint32_t cp = np + delta;
                        if (!bit(c.solid, cp) && crate_byte(s, cp) == 0) {
                            set_byte(cs, cb, cp);
                            cs.x = (cs.x & 0xFFFFFF00u) | np;
                            bool deadlocked = false;
                            for (int i = 0; i < c.nt; ++i) deadlocked |= bit(c.dead, get_byte(cs, 1 + i));
                            if (!deadlocked) {
                                valid = true;
                                ch = heuristic(c, cs);
                            }
                        }
                    }
                }
            }
            const unsigned vm = __ballot_sync(0xffffffffu, valid);
            const int nc = __popc(vm);
            uint32_t key = 0;
            if (valid) {
                const int idx = n_nodes + __popc(vm & ((1u << lane) - 1u));
                c.state[idx] = cs;
                c.meta[idx] = ((uint32_t)ch << 16) | (uint32_t)(d + 1);
                key = 2u * (uint32_t)ch + (uint32_t)bal2 * (uint32_t)(d + 1);
            }
            // lane 0 pushes the children in direction order; their keys come over by shuffle, not through memory
            for (int k = 0, rest = vm; k < nc; ++k, rest &= rest - 1) {
                const uint32_t kk = __shfl_sync(0xffffffffu, key, __ffs(rest) - 1);
                if (lane == 0) heap_push(heap, hn, (uint32_t)(n_nodes + k) | (kk << 16));
            }
            hn = __shfl_sync(0xffffffffu, hn, 0);
            n_nodes += nc;
            __syncwarp();
        }
        out_h = best_h;
        return false;
    }

    // ---- get_stats, part 1: counts, regions, solver preconditions (sokoban_prob.py:160-179) ---------------------
    // v[0..3] = player, crate, target, regions; v[4], v[5] = the defaults of dist-win / sol-length; v[6] = ratio.
    __device__ static bool prepare(const KParams& p, Ctx& c, const int8_t* grid, int lane, int (&v)[K]) {
        const int H = c.H, W = c.W;
        {
            uint4* st = (uint4*)c.stage;
            const uint4* src = (const uint4*)grid;
            for (int i = lane; i < p.row_stride / 16; i += 32) st[i] = src[i];
            __syncwarp();
        }
        int n_player = 0, n_crate = 0, n_target = 0;
        for (int i = lane; i < p.cells; i += 32) {
            const int t = c.stage[i];
            n_player += t == 2;
            n_crate += t == 3;
            n_target += t == 4;
        }
        n_player = __reduce_add_sync(0xffffffffu, n_player);
        n_crate = __reduce_add_sync(0xffffffffu, n_crate);
        n_target = __reduce_add_sync(0xffffffffu, n_target);
        uint16_t* rows = c.rows;
        for (int y = lane; y < H; y += 32) {
            uint32_t m = 0;
            for (int x = 0; x < W; ++x) m |= (uint32_t)(c.stage[y * W + x] != 1) << x;
            rows[y] = (uint16_t)m;
        }
        __syncwarp();
        const int regions = count_regions_rows(rows, 1, H, W, rows + 16, lane);
        v[0] = n_player;
        v[1] = n_crate;
        v[2] = n_target;
        v[3] = regions;
        v[4] = W * H * (W + H);                                         // sokoban_prob.py:171
        v[5] = 0;
        v[6] = abs(n_crate - n_target);
        return n_player == 1 && n_crate == n_target && n_crate > 0 && regions == 1;   // :174-179
    }

    // ---- the '#'-framed level of the staged grid (sokoban_prob.py:99-123, engine.py:137-186, 203-246) ----------
    __device__ static void frame_level(Ctx& c, int lane, uint4& root, int& root_h) {
        const int W = c.W, BW = c.BW, BH = c.BH;
        root = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
        int ncr = 0, ntg = 0;
        uint32_t player = 0;
        for (int w = 0; w < 8; ++w) {
            const int pidx = w * 32 + lane;
            int t = 1;
            if (pidx < BW * BH) {
                const int y = div_by(pidx, c.magic_bw), x = pidx - y * BW;
                if (x > 0 && y > 0 && x < BW - 1 && y < BH - 1) t = c.stage[(y - 1) * W + (x - 1)];
            }
            const unsigned sm = __ballot_sync(0xffffffffu, t == 1);
            const unsigned cm = __ballot_sync(0xffffffffu, t == 3);
            const unsigned tm = __ballot_sync(0xffffffffu, t == 4);
            const unsigned pm = __ballot_sync(0xffffffffu, t == 2);
            if (lane == 0) {
                c.solid[w] = sm;
                c.dead[w] = 0;
            }
            if (t == 3) c.cpos[ncr + __popc(cm & ((1u << lane) - 1u))] = (uint8_t)pidx;
            if (t == 4) c.tpos[ntg + __popc(tm & ((1u << lane) - 1u))] = (uint8_t)pidx;
            if (pm) player = w * 32 + (__ffs(pm) - 1);
            ncr += __popc(cm);
            ntg += __popc(tm);
        }
        __syncwarp();
        c.nt = ntg;
        root.x = (root.x & 0xFFFFFF00u) | player;
        for (int i = 0; i < ncr; ++i) set_byte(root, 1 + i, c.cpos[i]);
        __syncwarp();
        // static deadlocks (engine.py:203-246): non-target corners, and wall-hugging runs between two corners of
        // the same row / column
        uint32_t tmask[8];
#pragma unroll
        for (int w = 0; w < 8; ++w) tmask[w] = 0;
        for (int j = 0; j < ntg; ++j) tmask[c.tpos[j] >> 5] |= 1u << (c.tpos[j] & 31);
        for (int w = 0; w < 8; ++w) {
            const int pidx = w * 32 + lane;
            bool corner = false;
            if (pidx < BW * BH && !bit(c.solid, pidx)) {
                const bool up = bit(c.solid, pidx - BW), dn = bit(c.solid, pidx + BW), lf = bit(c.solid, pidx - 1),
                           rt = bit(c.solid, pidx + 1);
                corner = ((up && lf) || (up && rt) || (dn && lf) || (dn && rt)) && !((tmask[w] >> lane) & 1u);
            }
            const unsigned cm = __ballot_sync(0xffffffffu, corner);
            if (lane == 0) c.dead[w] = cm;
        }
        __syncwarp();
        uint32_t cornerm[8];
#pragma unroll
        for (int w = 0; w < 8; ++w) cornerm[w] = c.dead[w];
        __syncwarp();
        for (int pidx = lane; pidx < BW * BH; pidx += 32) {
            if (!((cornerm[pidx >> 5] >> (pidx & 31)) & 1u)) continue;
            // walk right, then down, from this corner; every further corner reached closes a run
            for (int dir = 0; dir < 2; ++dir) {
                const int step = dir == 0 ? 1 : BW;
                const int sa = dir == 0 ? BW : 1;     // the two sides that must hold a wall
                int q = pidx + step, last_corner = -1;
                while (!bit(c.solid, q) && !((tmask[q >> 5] >> (q & 31)) & 1u) &&
                       (bit(c.solid, q - sa) || bit(c.solid, q + sa))) {
                    if ((cornerm[q >> 5] >> (q & 31)) & 1u) last_corner = q;
                    q += step;
                }
                for (int r = pidx + step; r < last_corner; r += step) atomicOr(&c.dead[r >> 5], 1u << (r & 31));
            }
        }
        __syncwarp();
        root_h = heuristic(c, root);
    }

    __device__ static __forceinline__ uint32_t* jobs_hdr(const KParams& p) { return (uint32_t*)((uint8_t*)p.scratch + SokJobs::header); }
    __device__ static __forceinline__ int32_t* job_rec(const KParams& p, int j) {
        return (int32_t*)((uint8_t*)p.scratch + SokJobs::jobs) + (size_t)j * 8;
    }
    __device__ static __forceinline__ const int8_t* grid_of(const KParams& p, int64_t idx) {
        return (p.mode == MODE_STATS ? p.stats_grids : p.grids) + idx * p.row_stride;
    }
    // the final stats of a solved level go where phase D would have put them (lane 0)
    __device__ static void deliver(const KParams& p, int64_t idx, const int (&v)[K], const int32_t* old) {
        int32_t nw[K];
#pragma unroll
        for (int k = 0; k < K; ++k) nw[k] = v[k];
        if (p.mode == MODE_STATS) {
#pragma unroll
            for (int k = 0; k < K; ++k) p.stats_out[idx * K + k] = nw[k];
        } else {
            finish_env<K>(p, idx, nw, old);
        }
    }

    // pass 1 (inside k_step_search): everything but the solver; levels that need it become jobs
    __device__ static void stats(const KParams& p, Ctx& c, const int8_t* grid, int lane, int32_t* out) {
        int v[K];
        const bool run = prepare(p, c, grid, lane, v);
        if (run && v[1] > SOK_MAX_CRATES) {
            if (lane == 0 && p.status) atomicOr(p.status, 8);           // more crates than a packed state holds
        } else if (run) {
            const int64_t idx = (grid - grid_of(p, 0)) / p.row_stride;
            int slot = 0;
            if (lane == 0) slot = (int)atomicAdd(jobs_hdr(p), 1u);
            slot = __shfl_sync(0xffffffffu, slot, 0);
            if (slot < SokJobs::CAP) {
                if (lane == 0) {     // the job: which level, and (for a step) the stats the reward is measured from
                    int32_t* j = job_rec(p, slot);
                    j[0] = (int32_t)idx;
                    if (p.mode == MODE_STEP)
                        for (int k = 0; k < K; ++k) j[1 + k] = p.stats[idx * K + k];
                }
            } else {                 // list full: solve here, as before
                uint4 root;
                int root_h;
                frame_level(c, lane, root, root_h);
                run_game(c, root, root_h, lane, v);
            }
        }
        if (lane == 0)
            for (int k = 0; k < K; ++k) out[k] = v[k];
    }

    // _run_game (sokoban_prob.py:124-148), sequentially on one warp: BFS, then the A* passes if it hit the cap
    __device__ static void run_game(Ctx& c, const uint4 root, int root_h, int lane, int (&v)[K]) {
        int depth = 0, hbest = 0;
        bool exhausted = false;
        bool won = bfs_parallel(c, root, root_h, lane, depth, hbest, exhausted);
        if (!won && !exhausted)
            for (int mode = 1; mode <= 3 && !won; ++mode) won = search(c, root, root_h, mode, lane, depth, hbest, exhausted);
        if (won) {
            v[4] = 0;
            v[5] = depth;
        } else {
            v[4] = hbest;
        }
    }
};

// ------------------------------------------------------------------------------------------------
// pass 2: the BFS of every recorded level (persistent grid of warps, dynamic job counter)
// ------------------------------------------------------------------------------------------------
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) k_sokoban_solve(const KParams p, const int smem_per_warp) {
    using S = SokobanProb;
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    S::Ctx c = S::make_ctx(p, dyn_smem + (size_t)warp * smem_per_warp, blockIdx.x * WARPS + warp);
    uint32_t* hdr = S::jobs_hdr(p);
    const int n_jobs = (int)min(*(volatile uint32_t*)hdr, (uint32_t)SokJobs::CAP);
    int32_t* astar = (int32_t*)((uint8_t*)p.scratch + SokJobs::astar);
    for (;;) {
        int j = 0;
        if (lane == 0) j = (int)atomicAdd(hdr + 1, 1u);
        j = __shfl_sync(0xffffffffu, j, 0);
        if (j >= n_jobs) break;
        const int32_t* rec = S::job_rec(p, j);
        const int64_t idx = rec[0];
        int v[S::K];
        S::prepare(p, c, S::grid_of(p, idx), lane, v);
        uint4 root;
        int root_h;
        S::frame_level(c, lane, root, root_h);
        int depth = 0, hbest = 0;
        bool exhausted = false;
        const bool won = S::bfs_parallel(c, root, root_h, lane, depth, hbest, exhausted);
        if (won || exhausted) {
            v[4] = won ? 0 : hbest;
            v[5] = won ? depth : 0;
            if (lane == 0) S::deliver(p, idx, v, rec + 1);
        } else {
            // the BFS hit its iteration cap: three independent A* passes decide (pass 3), or here if that list is full
            int a = 0;
            if (lane == 0) a = (int)atomicAdd(hdr + 2, 1u);
            a = __shfl_sync(0xffffffffu, a, 0);
            if (a < SokJobs::ASTAR_CAP) {
                if (lane == 0) astar[a] = j;
            } else {
                bool w2 = false;
                for (int mode = 1; mode <= 3 && !w2; ++mode) w2 = S::search(c, root, root_h, mode, lane, depth, hbest, exhausted);
                v[4] = w2 ? 0 : hbest;
                v[5] = w2 ? depth : 0;
                if (lane == 0) S::deliver(p, idx, v, rec + 1);
            }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// pass 3: one A* pass per single-warp CTA, heap + visited table in shared memory
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_sokoban_astar(const KParams p, const int ctx_smem) {
    using S = SokobanProb;
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    const int lane = threadIdx.x;
    S::Ctx c = S::make_ctx(p, dyn_smem, blockIdx.x);
    uint32_t* heap = (uint32_t*)(dyn_smem + ctx_smem);
    uint16_t* table = (uint16_t*)(heap + SOK_NODES);
    const uint32_t* hdr = S::jobs_hdr(p);
    const int n_astar = (int)min(*(volatile const uint32_t*)(hdr + 2), (uint32_t)SokJobs::ASTAR_CAP);
    const int32_t* astar = (const int32_t*)((uint8_t*)p.scratch + SokJobs::astar);
    int32_t* results = (int32_t*)((uint8_t*)p.scratch + SokJobs::results);
    for (int i = blockIdx.x; i < 3 * n_astar; i += gridDim.x) {
        const int a = i / 3, mode = 1 + i - 3 * a;
        const int64_t idx = S::job_rec(p, astar[a])[0];
        int v[S::K];
        S::prepare(p, c, S::grid_of(p, idx), lane, v);
        uint4 root;
        int root_h;
        S::frame_level(c, lane, root, root_h);
        int depth = 0, hbest = 0;
        const bool won = S::astar_smem(c, root, root_h, mode, lane, heap, table, depth, hbest);
        if (lane == 0) {
            int32_t* r = results + ((size_t)a * 3 + (mode - 1)) * 4;
            r[0] = won;
            r[1] = depth;
            r[2] = hbest;
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// pass 4: first winning pass in the reference's order (balance 1, 0.5, 0), else the last pass's best heuristic
// (sokoban_prob.py:131-148); then re-arm the job lists for the next launch
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_sokoban_combine(const KParams p) {
    using S = SokobanProb;
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    const int lane = threadIdx.x;
    S::Ctx c = S::make_ctx(p, dyn_smem, 0);
    uint32_t* hdr = S::jobs_hdr(p);
    const int n_astar = (int)min(*(volatile uint32_t*)(hdr + 2), (uint32_t)SokJobs::ASTAR_CAP);
    const int32_t* astar = (const int32_t*)((uint8_t*)p.scratch + SokJobs::astar);
    const int32_t* results = (const int32_t*)((uint8_t*)p.scratch + SokJobs::results);
    for (int a = 0; a < n_astar; ++a) {
        const int32_t* rec = S::job_rec(p, astar[a]);
        const int64_t idx = rec[0];
        int v[S::K];
        S::prepare(p, c, S::grid_of(p, idx), lane, v);
        const int32_t* r = results + (size_t)a * 12;
        v[4] = r[2 * 4 + 2];
        for (int m = 0; m < 3; ++m)
            if (r[m * 4]) {
                v[4] = 0;
                v[5] = r[m * 4 + 1];
                break;
            }
        if (lane == 0) S::deliver(p, idx, v, rec + 1);
        __syncwarp();
    }
    __syncwarp();
    if (lane == 0) hdr[0] = hdr[1] = hdr[2] = hdr[3] = 0;
}

cudaError_t launch_sokoban(const KParams& p, cudaStream_t s, bool& supported) {
    supported = p.ndim == 2 && p.d0 <= 14 && p.d1 <= 14 && p.scratch != nullptr;
    if (!supported) return cudaSuccess;
    const int ctx_smem = SokobanProb::smem_bytes(p.row_stride);
    cudaError_t e = launch_search<SokobanProb>(p, s, ctx_smem, SOK_MAX_CTAS_PER_SM, SOK_MAX_CTAS);   // pass 1
    if (e != cudaSuccess || p.n_envs == 0) return e;
    int n_sm = 0;
    if ((e = sm_count(n_sm)) != cudaSuccess) return e;
    {   // pass 2: as many warps as pass 1 may hold (the per-warp scratch slices are shared by the two passes)
        auto k2 = k_sokoban_solve<SEARCH_WARPS>;
        const int dyn = ctx_smem * SEARCH_WARPS;
        if ((e = cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn)) != cudaSuccess) return e;
        const int ctas = std::min(n_sm * SOK_MAX_CTAS_PER_SM, SOK_MAX_CTAS);
        k2<<<ctas, SEARCH_WARPS * 32, dyn, s>>>(p, ctx_smem);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    {   // pass 3: one CTA per SM, the heap (40 008 x u32) and the table (32 768 x u16) in its shared memory
        const int ctx_al = (ctx_smem + 15) / 16 * 16;
        const int dyn = ctx_al + 4 * SOK_NODES + 2 * SokobanProb::ASTAR_TABLE;
        if ((e = cudaFuncSetAttribute(k_sokoban_astar, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn)) != cudaSuccess) return e;
        k_sokoban_astar<<<n_sm, 32, dyn, s>>>(p, ctx_al);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    k_sokoban_combine<<<1, 32, ctx_smem, s>>>(p);   // pass 4
    return cudaGetLastError();
}

}  // namespace pcgrl
