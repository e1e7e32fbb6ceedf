// smb (Super Mario Bros): fused env step with warp-per-grid get_stats, including the A* playthrough.
//
// Reference path replaced (paths relative to /root/reference/control_pcgrl/envs/):
//   probs/smb/smb_prob.py:132-154   get_stats (dist-floor, disjoint-tubes, enemies, empty, noise + play stats)
//   probs/smb/smb_prob.py:96-130    _run_game: level framing, A*(balance 1) then A*(balance 0), 10 000 iterations each
//   probs/smb/smb/engine.py:105-129 AStarAgent, :131-262 State (update physics, key, heuristic, win / lose)
//   helper.py:40-72 get_floor_dist, :74-121 get_type_grouping, :123-145 get_changes
//
// The level is the map with three extra columns on each side (smb_prob.py:99-113): rows above `H-3` are open
// and carry the exit marker in column W+4, row H-3 holds the player at x = 1 and a block at x = W+4, the last
// two rows are solid on both sides.  A node packs (x, y, airTime, last jump x, max jump gap) in one word and
// (jumps, depth) in another; jumps-dist (smb_prob.py:147-152) only needs the last jump x and the largest gap
// between consecutive jump x's, so the reference's jump_locs list is folded into those two numbers.
//
// Three launches per step (round 2; one warp per level for everything used to leave 20 of 32 lanes idle, with
// ~40 % of the instructions issued in lane 0's heap sifts):
//   1. k_step_search<SmbProb>: representation update, the map statistics and the framed level's solid bit map,
//      one warp per changed level; every changed level becomes a JOB (level index, old stats, map statistics,
//      bit map) in the global scratch.
//   2. k_smb_solve: the A* playthroughs, FOUR LANES PER LEVEL -- eight levels per warp.  A lane group's four
//      lanes are the four child directions of the popped node (engine.py:3); its first lane keeps the heap, so
//      the dependent heap walks of eight levels share one instruction stream.  Groups pull jobs from a global
//      counter as they finish.  Heap, node slots and the visited-key bit map of a group live in its slice of the
//      global scratch (L1 / L2 resident), the solid bit map in shared memory.  Node slots are recycled: the heap
//      array is kept as a permutation of the slot numbers -- positions below the heap size are the live entries,
//      positions above it the free slots -- so a group needs as many slots as its heap grows (1 900 on average
//      and < 3 200 on random levels, against 4 * 10 000 + 1 nodes when every pushed node keeps its slot).
//   3. k_smb_fallback: levels whose heap outgrew a group's slice (SMB_G_CAP entries), or maps whose bit map / visited-key map do
//      not fit a group's slices (SMB_G_SOLID words, SMB_G_VISITED bytes), are solved again by a whole warp with full-size slices (the
//      round-1 search); then the job lists are re-armed.  [116, 16] -- the reference's default, 116 rows of 16
//      columns (problem.py:31: height, width = map_shape) -- and [16, 116] both fit the groups.
//
// Exactness (SURVEY.md A-17, A-18): every pop counts as an iteration (also lose / already visited nodes); all
// four children are always pushed; the heap performs CPython's heappush / heappop moves with `<` on
// h + balance * depth only, because which of several equal-priority nodes is expanded first decides the
// jumps / jump positions that are reported.
#include "step_search.cuh"

namespace pcgrl {

constexpr int SMB_POWER = 10000;                 // smb_prob.py:21 _solver_power
constexpr int SMB_NODES = 4 * SMB_POWER + 8;
constexpr int SMB_WARPS = 8;             // warps per CTA
constexpr int SMB_MAX_CTAS_PER_SM = 4;   // A/B on B200 (116x16, 65 536 envs): 2 / 3 / 4 CTAs per SM -> 7.0 / 8.5 / 9.7e6 env-steps/s
constexpr int SMB_MAX_CTAS = 160 * SMB_MAX_CTAS_PER_SM;   // sizes the global scratch (>= 148 SMs x CTAs per SM)
constexpr int SMB_YOFF = 8;                      // y >= -5 (four rows per jump, re-jump possible from y = -1)

struct SmbScratch {
    static constexpr size_t nodes = 0;                                        // uint2[SMB_NODES]
    static constexpr size_t heap = nodes + sizeof(uint2) * (size_t)SMB_NODES; // u32[SMB_NODES]: idx | key << 16
    static constexpr size_t total = (heap + 4 * (size_t)SMB_NODES + 255) / 256 * 256;
};

// ---- jobs, per-group slices, fallback slices (in this order in the global scratch) --------------------------
constexpr int SMB_SOLVE_CTAS_PER_SM = 2;   // 64 lane groups x SMB_G_SMEM_WORDS words of shared memory per CTA = 112 KB
constexpr int SMB_G_CAP = 4096;                  // heap entries == node slots of one lane group
constexpr int SMB_G_SMEM_WORDS = 447;            // shared-memory words per lane group (heap top + bit map): 64 groups
                                                 // per CTA, two CTAs per SM
constexpr int SMB_G_SOLID = 128;                 // words of a group's shared-memory bit map: H * ceil((W + 6) / 32)
constexpr int SMB_G_VISITED = 5120;              // bytes of its visited-key map: (H + 8) * (W + 6)
constexpr int SMB_SOLVE_WARPS = 8;
constexpr int SMB_SOLVE_CTAS = 160 * SMB_SOLVE_CTAS_PER_SM;
constexpr int SMB_FALLBACK_CTAS = 160;
struct SmbJobs {
    static constexpr int CAP = 1 << 18;          // jobs per launch; launch_smb walks larger shards in ranges of CAP envs
    static constexpr int REC = 16;               // int32 per job: level index, old stats [9], map statistics [5]
    static constexpr int CLASSES = 4;            // predicted length: >= 1024, >= 512, >= 256 iterations, shorter / unknown
    static constexpr size_t header = 0;          // u32: [0] n_jobs [2] n_over [3] next over [4] CTAs done
                                                 //      [8..11] jobs per class [12..15] next job per class
    static constexpr size_t jobs = 256;
    static constexpr size_t solid = jobs + (size_t)CAP * REC * 4;              // u32[CAP][SMB_G_SOLID]
    static constexpr size_t over = solid + (size_t)CAP * SMB_G_SOLID * 4;      // int32[CAP]: jobs for the fallback
    static constexpr size_t cls = over + (size_t)CAP * 4;                      // int32[CLASSES][CAP]: job numbers
    static constexpr size_t total = (cls + (size_t)CLASSES * CAP * 4 + 255) / 256 * 256;
};
// shared-memory words of one lane group: bit map + heap top.  The count is odd so that the eight group leaders of a
// warp, who walk their heaps in step, touch eight different banks.
__host__ __device__ inline int smb_group_heap_words(int H, int W) { return SMB_G_SMEM_WORDS - H * ((W + 6 + 31) / 32); }
struct SmbGroupScratch {
    static constexpr size_t nodes = 0;                                         // uint2[SMB_G_CAP]
    static constexpr size_t heap = nodes + 8 * (size_t)SMB_G_CAP;              // u32[SMB_G_CAP]: slot | key << 16
    static constexpr size_t visited = heap + 4 * (size_t)SMB_G_CAP;            // u8[SMB_G_VISITED]
    static constexpr size_t total = (visited + (size_t)SMB_G_VISITED + 255) / 256 * 256;
};
constexpr size_t SMB_GROUPS_BYTES = SmbGroupScratch::total * (size_t)SMB_SOLVE_CTAS * SMB_SOLVE_WARPS * 8;

// ... and behind them int32[n_envs]: the iterations each env's last playthrough took.  A step's time is bounded below
// by its longest playthrough (a chain of dependent heap operations: ~1 us per iteration, up to 2 x 10 000 iterations),
// so the lane groups take the jobs longest-predicted first; one edited tile rarely changes the length class.
constexpr size_t SMB_HIST_OFF = SmbJobs::total + SMB_GROUPS_BYTES + SmbScratch::total * (size_t)SMB_FALLBACK_CTAS * SMB_WARPS;
int64_t smb_scratch_bytes(int64_t n_envs) { return (int64_t)(SMB_HIST_OFF + (size_t)(n_envs > 0 ? n_envs : 0) * 4 + 256); }

struct SmbLayout {
    int stage, solid, visited, total, visited_bytes;
};
__host__ __device__ inline SmbLayout smb_layout(int H, int W, int row_stride) {
    SmbLayout L;
    int o = 0;
    L.stage = o;   o += (row_stride + 15) / 16 * 16;
    L.solid = o;   o += (H * ((W + 6 + 31) / 32) * 4 + 15) / 16 * 16;   // RW = ceil((W + 6) / 32) words per row
    L.visited_bytes = ((H + SMB_YOFF) * (W + 6) + 15) / 16 * 16;   // 8 airTime slots per (x, y) = one byte
    L.visited = o; o += L.visited_bytes;
    L.total = (o + 15) / 16 * 16;
    return L;
}

struct SmbProb {
    static constexpr int K = 9;   // dist-floor disjoint-tubes enemies empty noise jumps jumps-dist dist-win sol-length

    struct Ctx {
        int H, W, LW, RW, exit_x, visited_bytes;
        uint8_t* stage;
        uint32_t* solid;     // [H][RW]
        uint8_t* visited;    // [(y + YOFF) * LW + x] bit airTime
        uint2* nodes;
        uint32_t* heap;
    };

    __device__ static Ctx make_ctx(const KParams& p, uint8_t* ws, int global_warp) {
        Ctx c;
        c.H = p.d0; c.W = p.d1;
        c.LW = c.W + 6;
        c.RW = (c.LW + 31) >> 5;
        c.exit_x = c.W + 4;
        const SmbLayout L = smb_layout(c.H, c.W, p.row_stride);
        c.stage = ws + L.stage;
        c.solid = (uint32_t*)(ws + L.solid);
        c.visited = ws + L.visited;
        c.visited_bytes = L.visited_bytes;
        // full-size node pool / heap: only the fallback's warps search with them (global_warp < its warp count)
        uint8_t* g = (uint8_t*)p.scratch + SmbJobs::total + SMB_GROUPS_BYTES +
                     (size_t)(global_warp % (SMB_FALLBACK_CTAS * SMB_WARPS)) * SmbScratch::total;
        c.nodes = (uint2*)(g + SmbScratch::nodes);
        c.heap = (uint32_t*)(g + SmbScratch::heap);
        return c;
    }

    __device__ static __forceinline__ bool solid_at(const Ctx& c, int x, int y) {
        return (c.solid[y * c.RW + (x >> 5)] >> (x & 31)) & 1u;
    }
    // engine.py:190-193 checkMovableLocation
    __device__ static __forceinline__ bool movable(const Ctx& c, int x, int y) {
        if (y < 0) return true;
        return !(x < 0 || x >= c.LW || y >= c.H || solid_at(c, x, y));
    }

    struct Node {
        int x, y, air, last_jx, gap, jumps, depth;
    };
    __device__ static __forceinline__ uint2 pack(const Node& n) {
        return make_uint2((uint32_t)n.x | ((uint32_t)(n.y + SMB_YOFF) << 7) | ((uint32_t)n.air << 15) |
                              ((uint32_t)n.last_jx << 18) | ((uint32_t)n.gap << 25),
                          (uint32_t)n.jumps | ((uint32_t)n.depth << 16));
    }
    __device__ static __forceinline__ Node unpack(const uint2 v) {
        Node n;
        n.x = v.x & 0x7F;
        n.y = (int)((v.x >> 7) & 0xFF) - SMB_YOFF;
        n.air = (v.x >> 15) & 0x7;
        n.last_jx = (v.x >> 18) & 0x7F;
        n.gap = (v.x >> 25) & 0x7F;
        n.jumps = v.y & 0xFFFF;
        n.depth = v.y >> 16;
        return n;
    }

    // engine.py:195-237 State.update for a node that is neither won nor lost
    __device__ static __forceinline__ Node update(const Ctx& c, Node n, int dx, int dy) {
        bool ground = false;
        if (n.y < c.H - 1 && n.y >= -1) ground = solid_at(c, n.x, n.y + 1);
        int nx = n.x, ny = n.y;
        if (dx != 0 && movable(c, nx + dx, ny)) nx += dx;
        if (dy == -1) {
            if (ground && movable(c, nx, ny - 1)) {
                n.air = 5;
                n.jumps += 1;
                n.gap = max(n.gap, n.x - n.last_jx);   // jump_locs.append((x, y)) with the pre-move x
                n.last_jx = n.x;
            }
        } else if (n.air > 0) {
            n.air = 1;
        }
        if (n.air > 1) {
            n.air -= 1;
            if (movable(c, nx, ny - 1)) ny -= 1;
            else n.air = 1;
        } else if (n.air == 1) {
            n.air = 0;
        } else if (movable(c, nx, ny + 1)) {
            ny += 1;
        }
        n.x = nx;
        n.y = ny;
        n.depth += 1;
        return n;
    }

    // CPython heapq on (key << 16 | idx) entries (lane 0 only); see step_sokoban.cu
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

    // engine.py:105-129 AStarAgent.getSolution.  Returns true on win; `res` = winning node or the best node.
    __device__ static bool search(Ctx& c, int balance, int lane, Node& res) {
        for (int i = lane; i < c.visited_bytes / 16; i += 32) ((uint4*)c.visited)[i] = make_uint4(0, 0, 0, 0);
        Node root;
        root.x = 1; root.y = c.H - 3; root.air = 0; root.last_jx = 0; root.gap = 0; root.jumps = 0; root.depth = 0;
        if (lane == 0) {
            c.nodes[0] = pack(root);
            c.heap[0] = (uint32_t)(c.exit_x - root.x) << 16;
        }
        __syncwarp();
        int n_nodes = 1, hn = 1, iters = 0;
        int best_h = 0x7FFFFFFF, best_d = 0;
        Node best = root;
        const int dx = lane & 1, dy = (lane & 2) ? -1 : 0;       // engine.py:3: (0,0) (1,0) (0,-1) (1,-1)
        while (iters < SMB_POWER && hn > 0) {
            ++iters;
            int cur = 0;
            if (lane == 0) cur = (int)(heap_pop(c.heap, hn) & 0xFFFFu);
            cur = __shfl_sync(0xffffffffu, cur, 0);
            hn = __shfl_sync(0xffffffffu, hn, 0);
            const Node n = unpack(c.nodes[cur]);
            if (n.y >= c.H) continue;                             // checkLose: skipped, still an iteration
            if (n.x >= c.exit_x) {                                // checkWin
                res = n;
                return true;
            }
            const int vidx = (n.y + SMB_YOFF) * c.LW + n.x;
            const uint32_t vb = c.visited[vidx];
            if ((vb >> n.air) & 1u) continue;
            const int h = c.exit_x - n.x;
            if (h < best_h || (h == best_h && n.depth < best_d)) {
                best_h = h;
                best_d = n.depth;
                best = n;
            }
            uint32_t key = 0;
            if (lane == 0) c.visited[vidx] = (uint8_t)(vb | (1u << n.air));
            if (lane < 4) {
                const Node ch = update(c, n, dx, dy);
                c.nodes[n_nodes + lane] = pack(ch);
                key = (uint32_t)((c.exit_x - ch.x) + balance * ch.depth);
            }
            // heap pushes in direction order (lane 0), keys fetched by shuffle
            for (int k = 0; k < 4; ++k) {
                const uint32_t kk = __shfl_sync(0xffffffffu, key, k);
                if (lane == 0) {
                    c.heap[hn] = (uint32_t)(n_nodes + k) | (kk << 16);
                    sift_down(c.heap, 0, hn);
                    ++hn;
                }
            }
            hn = __shfl_sync(0xffffffffu, hn, 0);
            n_nodes += 4;
            __syncwarp();
        }
        res = best;
        return false;
    }

    // map statistics of a staged grid whose width is a multiple of four, four tiles per word (byte-wise SIMD compares)
    __device__ static __forceinline__ void map_stats_words(const KParams& p, const Ctx& c, int lane, int& dist_floor, int& tubes,
                                                           int& enemies, int& empty, int& noise) {
        const int H = c.H, W = c.W, WW = W >> 2;
        const uint8_t* g = c.stage;
        const uint32_t* gw = (const uint32_t*)c.stage;
        const uint32_t magic_ww = div_magic(WW);
        for (int i = lane; i < (p.cells >> 2); i += 32) {
            const uint32_t w = gw[i];
            const int y = div_by(i, magic_ww), xw = i - y * WW;
            empty += __popc(__vcmpeq4(w, 0u)) >> 3;
            // helper.py:123 get_changes: every tile against its left and its upper neighbour
            const uint32_t left = (w << 8) | (xw ? gw[i - 1] >> 24 : (w & 0xFFu));
            noise += __popc(__vcmpne4(w, left)) >> 3;
            if (y > 0) noise += __popc(__vcmpne4(w, gw[i - WW])) >> 3;
            enemies += __popc(__vcmpeq4(w, 0x02020202u)) >> 3;
            for (uint32_t m = __vcmpeq4(w, 0x06060606u); m;) {   // helper.py:103 tubes with exactly one tube beside
                const int b = (__ffs(m) - 1) >> 3, cell = i * 4 + b, x = xw * 4 + b;
                m &= ~(0xFFu << (8 * b));
                const int nb = (x > 0 && g[cell - 1] == 6) + (x < W - 1 && g[cell + 1] == 6);
                tubes += nb == 1;
            }
        }
        // helper.py:40-46: every enemy's distance to the first floor tile below it (H - 1 when there is none).  One lane
        // per column walks it bottom-up remembering the nearest floor row -- a scan per enemy (265 enemies on a
        // uniform-random [116, 16] map) was half of this kernel's instructions at 3-5 lanes
        for (int x = lane; x < W; x += 32) {
            int nf = -1;
            for (int y = H - 1; y >= 0; --y) {
                const int t = g[y * W + x];
                if (t == 2) dist_floor += nf < 0 ? H - 1 : nf - y - 1;
                if (t == 1 || t == 3 || t == 4) nf = y;
            }
        }
    }

    // map statistics (smb_prob.py:134-139) and the framed level's solid bit map in c.solid; whole warp
    __device__ static void map_stats(const KParams& p, Ctx& c, const int8_t* grid, int lane, int (&v)[5]) {
        const int H = c.H, W = c.W;
        {
            uint4* st = (uint4*)c.stage;
            const uint4* src = (const uint4*)grid;
            for (int i = lane; i < p.row_stride / 16; i += 32) st[i] = src[i];
            __syncwarp();
        }
        const uint8_t* g = c.stage;
        int dist_floor = 0, tubes = 0, enemies = 0, empty = 0, noise = 0;
        if ((W & 3) == 0) {
            map_stats_words(p, c, lane, dist_floor, tubes, enemies, empty, noise);
        } else {
        const uint32_t magic_w = div_magic(W);
        for (int i = lane; i < p.cells; i += 32) {
            const int y = div_by(i, magic_w), x = i - y * W, t = g[i];
            empty += t == 0;
            if (t == 2) {                                        // helper.py:40-46 distance of an enemy to the floor
                ++enemies;
                int d = H - 1;
                for (int dy = 1; y + dy < H; ++dy) {
                    const int f = g[i + dy * W];
                    if (f == 1 || f == 3 || f == 4) {
                        d = dy - 1;
                        break;
                    }
                }
                dist_floor += d;
            }
            if (t == 6) {                                        // helper.py:103 tubes with exactly one tube beside
                const int nb = (x > 0 && g[i - 1] == 6) + (x < W - 1 && g[i + 1] == 6);
                tubes += nb == 1;
            }
            noise += (x > 0 && g[i - 1] != t) + (y > 0 && g[i - W] != t);   // helper.py:123 get_changes h + v
        }
        }
        v[0] = __reduce_add_sync(0xffffffffu, dist_floor);
        v[1] = __reduce_add_sync(0xffffffffu, tubes);
        v[2] = __reduce_add_sync(0xffffffffu, enemies);
        v[3] = __reduce_add_sync(0xffffffffu, empty);
        v[4] = __reduce_add_sync(0xffffffffu, noise);

        // the framed level's solid bit map (smb_prob.py:96-113; " # ## #": codes 1, 3, 4, 6 are solid)
        for (int y = lane; y < H; y += 32) {
            uint32_t w[4] = {0, 0, 0, 0};
            if ((W & 3) == 0) {
                // four tiles per word: solid <=> bit 0 != bit 2 of the code; the four flag bits are gathered into a
                // nibble by one multiply (bit 8j lands on 24 + j, the cross terms stay below bit 24)
                const uint32_t* gw = (const uint32_t*)g + y * (W >> 2);
                for (int k = 0; k < (W >> 2); ++k) {
                    const uint32_t t4 = gw[k];
                    const uint32_t nib = ((((t4 ^ (t4 >> 2)) & 0x01010101u) * 0x01020408u) >> 24) & 0xFu;
                    const int bit = 4 * k + 3;
                    const uint64_t sh = (uint64_t)nib << (bit & 31);
                    w[bit >> 5] |= (uint32_t)sh;
                    if ((bit >> 5) < 3) w[(bit >> 5) + 1] |= (uint32_t)(sh >> 32);
                }
            } else {
            for (int x = 0; x < W; ++x) {
                const int t = g[y * W + x];
                if (t == 1 || t == 3 || t == 4 || t == 6) w[(x + 3) >> 5] |= 1u << ((x + 3) & 31);
            }
            }
            if (y == H - 3) {
                w[(W + 4) >> 5] |= 1u << ((W + 4) & 31);
            } else if (y > H - 3) {
                w[0] |= 7u;
                for (int x = W + 3; x < W + 6; ++x) w[x >> 5] |= 1u << (x & 31);
            }
            for (int k = 0; k < c.RW; ++k) c.solid[y * c.RW + k] = w[k];
        }
        __syncwarp();
    }

    // the play statistics of the search's result node (smb_prob.py:144-153)
    __device__ static __forceinline__ void play_stats(int W, int exit_x, const Node& res, bool won, int32_t* out) {
        out[5] = res.jumps;
        out[6] = max(res.gap, W - res.last_jx);                  // smb_prob.py:147-152 with _width = map_shape[1]
        out[7] = won ? 0 : exit_x - res.x;
        out[8] = won ? res.depth : 0;
    }

    // get_stats on one warp with the full-size slices (the fallback; round 1's only path)
    __device__ static void stats_full(const KParams& p, Ctx& c, const int8_t* grid, int lane, int32_t (&out)[K]) {
        int v[5];
        map_stats(p, c, grid, lane, v);
        // _run_game (smb_prob.py:115-130)
        Node res;
        bool won = search(c, 1, lane, res);
        if (!won) {
            __syncwarp();
            won = search(c, 0, lane, res);
        }
        for (int k = 0; k < 5; ++k) out[k] = v[k];
        play_stats(c.W, c.exit_x, res, won, out);
        __syncwarp();
    }

    // maps a lane group can play: bit map and visited-key map fit its slices
    __host__ __device__ static bool groups_fit(int H, int W) {
        return H * ((W + 6 + 31) / 32) <= SMB_G_SOLID && (H + SMB_YOFF) * (W + 6) + 15 <= SMB_G_VISITED &&
               smb_group_heap_words(H, W) >= 64;
    }
    __device__ static __forceinline__ uint32_t* jobs_hdr(const KParams& p) { return (uint32_t*)((uint8_t*)p.scratch + SmbJobs::header); }
    __device__ static __forceinline__ int32_t* job_rec(const KParams& p, int j) {
        return (int32_t*)((uint8_t*)p.scratch + SmbJobs::jobs) + (size_t)j * SmbJobs::REC;
    }
    __device__ static __forceinline__ uint32_t* job_solid(const KParams& p, int j) {
        return (uint32_t*)((uint8_t*)p.scratch + SmbJobs::solid) + (size_t)j * SMB_G_SOLID;
    }
    __device__ static __forceinline__ int32_t* job_class(const KParams& p, int k) {
        return (int32_t*)((uint8_t*)p.scratch + SmbJobs::cls) + (size_t)k * SmbJobs::CAP;
    }
    __device__ static __forceinline__ int32_t* history(const KParams& p) { return (int32_t*)((uint8_t*)p.scratch + SMB_HIST_OFF); }
    __device__ static __forceinline__ const int8_t* grid_of(const KParams& p, int64_t idx) {
        return (p.mode == MODE_STATS ? p.stats_grids : p.grids) + idx * p.row_stride;
    }
    // the final stats of a played level go where phase D would have put them (one lane)
    __device__ static void deliver(const KParams& p, int64_t idx, const int32_t (&nw)[K], const int32_t* old) {
        if (p.mode == MODE_STATS) {
#pragma unroll
            for (int k = 0; k < K; ++k) p.stats_out[idx * K + k] = nw[k];
        } else {
            finish_env<K>(p, idx, nw, old);
        }
    }

    // pass 1 (inside k_step_search): map statistics + bit map; the playthrough becomes a job.  The provisional
    // stats phase D stores (and the reward it computes from them) are replaced when the job is delivered.
    __device__ static void stats(const KParams& p, Ctx& c, const int8_t* grid, int lane, int32_t* out) {
        int v[5];
        map_stats(p, c, grid, lane, v);
        const int64_t idx = (grid - grid_of(p, 0)) / p.row_stride;
        int slot = 0;
        if (lane == 0) {
            slot = (int)atomicAdd(jobs_hdr(p), 1u);              // < CAP: launch_smb hands pass 1 at most CAP envs
            const int pred = p.mode == MODE_STATS ? 0 : history(p)[idx];
            const int k = pred >= 1024 ? 0 : (pred >= 512 ? 1 : (pred >= 256 ? 2 : 3));
            job_class(p, k)[atomicAdd(jobs_hdr(p) + 8 + k, 1u)] = slot;
        }
        slot = __shfl_sync(0xffffffffu, slot, 0);
        int32_t* j = job_rec(p, slot);
        if (lane == 0) j[0] = (int32_t)idx;
        if (lane < K && p.mode == MODE_STEP) j[1 + lane] = p.stats[idx * K + lane];
        if (lane < 5) j[1 + K + lane] = v[lane];
        if (groups_fit(c.H, c.W)) {
            uint32_t* sd = job_solid(p, slot);
            for (int i = lane; i < c.H * c.RW; i += 32) sd[i] = c.solid[i];
        }
        if (lane < K) out[lane] = lane < 5 ? v[lane] : 0;
        __syncwarp();
    }
};

// ------------------------------------------------------------------------------------------------
// pass 2: the playthroughs, four lanes per level (see the head of this file)
// ------------------------------------------------------------------------------------------------
// A group's heap: the first SMB_G_SH positions (the top levels -- all of it for the heaps of a few hundred entries
// that [116, 16] levels grow) in shared memory, the rest in its global slice.  Walking the heap is a chain of
// dependent loads; from L2 that chain was ~90 % of a playthrough's time.
// HYBRID = false: the whole heap is the shared-memory part (narrow levels; a heap that outgrows it goes to the fallback).
template <bool HYBRID>
struct SmbGroupHeap {
    uint32_t* sh;
    uint32_t* gl;
    int n_sh;
    __device__ __forceinline__ uint32_t* at(int i) const { return (!HYBRID || i < n_sh) ? sh + i : gl + i; }
};
// heapq._siftdown (the walk towards the root after a push / at the end of a pop)
template <bool HYBRID>
__device__ __forceinline__ void smb_sift_down(const SmbGroupHeap<HYBRID>& hp, int start, int pos) {
    const uint32_t item = *hp.at(pos);
    while (pos > start) {
        const int parent = (pos - 1) >> 1;
        const uint32_t pe = *hp.at(parent);
        if ((item >> 16) < (pe >> 16)) {
            *hp.at(pos) = pe;
            pos = parent;
            continue;
        }
        break;
    }
    *hp.at(pos) = item;
}
// CPython's heappop on a heap of n entries that also keeps the free slots: the popped entry's slot is parked at
// position n - 1, the first position above the shrunken heap.  Returns the popped node's slot.
template <bool HYBRID>
__device__ __forceinline__ uint32_t smb_pop_recycle(const SmbGroupHeap<HYBRID>& hp, int n) {
    const int m = n - 1;
    const uint32_t last = *hp.at(m);
    uint32_t ret = last;
    if (m > 0) {
        ret = *hp.at(0);
        int pos = 0, child = 1;
        while (child < m) {
            const int right = child + 1;
            uint32_t ce = *hp.at(child);
            if (right < m) {
                const uint32_t re = *hp.at(right);
                if (!((ce >> 16) < (re >> 16))) {
                    child = right;
                    ce = re;
                }
            }
            *hp.at(pos) = ce;
            pos = child;
            child = 2 * pos + 1;
        }
        *hp.at(pos) = last;
        smb_sift_down(hp, 0, pos);
    }
    *hp.at(m) = ret;
    return ret & 0xFFFFu;
}

template <int WARPS, bool HYBRID>
__global__ void __launch_bounds__(WARPS * 32) k_smb_solve(const KParams p, const int g_cap) {
    using S = SmbProb;
    constexpr int K = S::K;
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane & 3, gbase = lane & ~3;
    const unsigned gmask = 0xFu << gbase;
    const int g_local = warp * 8 + (lane >> 2);
    S::Ctx c;
    c.H = p.d0; c.W = p.d1;
    c.LW = c.W + 6;
    c.RW = (c.LW + 31) >> 5;
    c.exit_x = c.W + 4;
    uint32_t* g_smem = (uint32_t*)dyn_smem + g_local * SMB_G_SMEM_WORDS;
    c.solid = g_smem;
    c.visited_bytes = ((c.H + SMB_YOFF) * c.LW + 15) / 16 * 16;
    uint8_t* gs = (uint8_t*)p.scratch + SmbJobs::total +
                  ((size_t)blockIdx.x * (WARPS * 8) + g_local) * SmbGroupScratch::total;
    c.nodes = (uint2*)(gs + SmbGroupScratch::nodes);
    c.heap = (uint32_t*)(gs + SmbGroupScratch::heap);
    c.visited = gs + SmbGroupScratch::visited;
    c.stage = nullptr;
    SmbGroupHeap<HYBRID> hp;
    hp.sh = g_smem + c.H * c.RW;
    hp.gl = c.heap;
    hp.n_sh = smb_group_heap_words(c.H, c.W);
    uint32_t* hdr = S::jobs_hdr(p);
    int32_t* over = (int32_t*)((uint8_t*)p.scratch + SmbJobs::over);
    int cls = 0, iters_job = 0;                                  // class this group draws from; iterations of its job so far
    const int dx = sub & 1, dy = (sub & 2) ? -1 : 0;             // engine.py:3: (0,0) (1,0) (0,-1) (1,-1)

    S::Node root;
    root.x = 1; root.y = c.H - 3; root.air = 0; root.last_jx = 0; root.gap = 0; root.jumps = 0; root.depth = 0;
    // group state, identical in the group's four lanes.  0: wants a job, 1: searching, 2: the list is empty
    int state = 0, job = 0, balance = 1, start = 0;
    int iters = 0, hn = 0, hw = 0, best_h = 0, best_d = 0;
    S::Node best = root;
    for (;;) {
        if (state == 0) {
            int j = -1;
            if (sub == 0) {                                      // longest-predicted class first
                for (; cls < SmbJobs::CLASSES; ++cls) {
                    const uint32_t n_k = *(volatile uint32_t*)(hdr + 8 + cls);
                    if (n_k == 0) continue;
                    const uint32_t t = atomicAdd(hdr + 12 + cls, 1u);
                    if (t < n_k) {
                        j = S::job_class(p, cls)[t];
                        break;
                    }
                }
            }
            j = __shfl_sync(gmask, j, gbase);
            cls = __shfl_sync(gmask, cls, gbase);
            if (j < 0) {
                state = 2;
            } else {
                job = j;
                iters_job = 0;
                const uint32_t* src = S::job_solid(p, j);
                for (int i = sub; i < c.H * c.RW; i += 4) c.solid[i] = src[i];
                balance = 1;
                start = 1;
                state = 1;
            }
        }
        if (__all_sync(0xffffffffu, state == 2)) break;          // the whole warp meets here once per round
        if (state == 1 && start) {                               // engine.py:105-112: a fresh search
            for (int i = sub; i < c.visited_bytes / 16; i += 4) ((uint4*)c.visited)[i] = make_uint4(0, 0, 0, 0);
            if (sub == 0) {
                c.nodes[0] = S::pack(root);
                *hp.at(0) = (uint32_t)(c.exit_x - root.x) << 16;
            }
            iters = 0;
            hn = 1;
            hw = 1;
            best_h = 0x7FFFFFFF;
            best_d = 0;
            best = root;
            start = 0;
            __syncwarp(gmask);
        } else if (state == 1) {
            bool finished = false, won = false;
            S::Node res = best;
            if (iters >= SMB_POWER || hn == 0) {
                finished = true;
            } else {
                ++iters;
                // the pop returns the heap's root: its node (L2) is requested before the leader walks the heap
                const uint32_t cur = *hp.at(0) & 0xFFFFu;
                __syncwarp(gmask);                               // the group has read the root before the leader rewrites it
                const uint2 packed = c.nodes[cur];
                if (sub == 0) smb_pop_recycle(hp, hn);
                --hn;
                const S::Node n = S::unpack(packed);
                if (n.y >= c.H) {
                    // checkLose: skipped, still an iteration
                } else if (n.x >= c.exit_x) {                    // checkWin
                    finished = true;
                    won = true;
                    res = n;
                } else {
                    const int vidx = (n.y + SMB_YOFF) * c.LW + n.x;
                    const uint32_t vb = c.visited[vidx];
                    if (!((vb >> n.air) & 1u)) {
                        const int h = c.exit_x - n.x;
                        if (h < best_h || (h == best_h && n.depth < best_d)) {
                            best_h = h;
                            best_d = n.depth;
                            best = n;
                        }
                        if (hn + 4 > g_cap) {                    // the heap outgrows this group's slice: fallback
                            if (sub == 0) over[atomicAdd(hdr + 2, 1u)] = job;
                            state = 0;
                        } else {
                            __syncwarp(gmask);                   // every lane has read the node and the visited byte
                            if (sub == 0) c.visited[vidx] = (uint8_t)(vb | (1u << n.air));
                            const int pos = hn + sub;            // child k takes the slot parked at position hn + k
                            const uint32_t slot = pos < hw ? (*hp.at(pos) & 0xFFFFu) : (uint32_t)pos;
                            const S::Node ch = S::update(c, n, dx, dy);
                            c.nodes[slot] = S::pack(ch);
                            const uint32_t entry = slot | ((uint32_t)((c.exit_x - ch.x) + balance * ch.depth) << 16);
#pragma unroll
                            for (int k = 0; k < 4; ++k) {        // heap pushes in direction order
                                const uint32_t e = __shfl_sync(gmask, entry, gbase + k);
                                if (sub == 0) {
                                    *hp.at(hn + k) = e;
                                    smb_sift_down(hp, 0, hn + k);
                                }
                            }
                            hn += 4;
                            hw = max(hw, hn);
                        }
                    }
                }
                __syncwarp(gmask);
            }
            if (finished) {
                iters_job += iters;
                if (!won && balance == 1) {                      // smb_prob.py:121-127: second pass with balance 0
                    balance = 0;
                    start = 1;
                } else {
                    if (sub == 0) {
                        const int32_t* rec = S::job_rec(p, job);
                        int32_t out[K];
#pragma unroll
                        for (int k = 0; k < 5; ++k) out[k] = rec[1 + K + k];
                        S::play_stats(c.W, c.exit_x, res, won, out);
                        S::deliver(p, rec[0], out, rec + 1);
                        if (p.mode != MODE_STATS) S::history(p)[rec[0]] = iters_job;
                    }
                    state = 0;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// pass 3: jobs the lane groups gave up (or every job when the map is taller than their bit map), one warp each,
// with the full-size slices; the last CTA re-arms the lists
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SMB_WARPS * 32) k_smb_fallback(const KParams p, const int smem_per_warp, const int all_jobs) {
    using S = SmbProb;
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    S::Ctx c = S::make_ctx(p, dyn_smem + (size_t)warp * smem_per_warp, blockIdx.x * SMB_WARPS + warp);
    uint32_t* hdr = S::jobs_hdr(p);
    const int n_jobs = (int)min(*(volatile uint32_t*)hdr, (uint32_t)SmbJobs::CAP);
    const int n = all_jobs ? n_jobs : (int)min(*(volatile uint32_t*)(hdr + 2), (uint32_t)SmbJobs::CAP);
    const int32_t* over = (const int32_t*)((uint8_t*)p.scratch + SmbJobs::over);
    for (;;) {
        int i = 0;
        if (lane == 0) i = (int)atomicAdd(hdr + 3, 1u);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= n) break;
        const int32_t* rec = S::job_rec(p, all_jobs ? i : over[i]);
        int32_t out[S::K];
        S::stats_full(p, c, S::grid_of(p, rec[0]), lane, out);
        if (lane == 0) S::deliver(p, rec[0], out, rec + 1);
        __syncwarp();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(hdr + 4, 1u) == gridDim.x - 1) {
            for (int i = 0; i < 16; ++i) hdr[i] = 0;
            __threadfence();
        }
    }
}

cudaError_t launch_smb(const KParams& p, cudaStream_t s, bool& supported, int& n_launches) {
    // level width W + 6 <= 128 (7-bit x), H + 8 <= 255, at least one open row above the player's
    supported = p.ndim == 2 && p.d1 <= 122 && p.d0 >= 4 && p.d0 <= 240 && p.scratch != nullptr;
    n_launches = 0;
    if (!supported) return cudaSuccess;
    const SmbLayout L = smb_layout(p.d0, p.d1, p.row_stride);
    if (L.total * SMB_WARPS > 200 * 1024) {
        supported = false;
        return cudaSuccess;
    }
    int n_sm = 0;
    cudaError_t e;
    if ((e = sm_count(n_sm)) != cudaSuccess) return e;
    const char* cap_env = getenv("PCGRL_SMB_GROUP_CAP");         // tests shrink it to drive levels into the fallback
    // narrow levels ([116, 16]: heaps of 30-270 entries) keep the whole heap in shared memory; wide ones ([16, 116]:
    // ~1 900) continue in the group's global slice
    const bool hybrid = p.d1 + 6 > 32;
    const int cap_max = hybrid ? SMB_G_CAP : smb_group_heap_words(p.d0, p.d1);
    const int g_cap = cap_env ? std::min(std::max(atoi(cap_env), 8), cap_max) : cap_max;
    const bool groups = SmbProb::groups_fit(p.d0, p.d1);
    for (int64_t lo = 0; lo < p.n_envs; lo += SmbJobs::CAP) {
        const int64_t hi = std::min<int64_t>(p.n_envs, lo + SmbJobs::CAP);
        if ((e = launch_search<SmbProb, SMB_WARPS>(p, s, L.total, SMB_MAX_CTAS_PER_SM, SMB_MAX_CTAS, lo, hi)) != cudaSuccess) return e;
        ++n_launches;
        if (groups) {
            auto k2 = hybrid ? k_smb_solve<SMB_SOLVE_WARPS, true> : k_smb_solve<SMB_SOLVE_WARPS, false>;
            const int dyn = SMB_SOLVE_WARPS * 8 * SMB_G_SMEM_WORDS * 4;
            if ((e = cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn)) != cudaSuccess) return e;
            const int ctas = std::min(n_sm * SMB_SOLVE_CTAS_PER_SM, SMB_SOLVE_CTAS);
            k2<<<ctas, SMB_SOLVE_WARPS * 32, dyn, s>>>(p, g_cap);
            if ((e = cudaGetLastError()) != cudaSuccess) return e;
            ++n_launches;
        }
        const int dyn = L.total * SMB_WARPS;
        if ((e = cudaFuncSetAttribute(k_smb_fallback, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn)) != cudaSuccess) return e;
        k_smb_fallback<<<std::min(n_sm, SMB_FALLBACK_CTAS), SMB_WARPS * 32, dyn, s>>>(p, L.total, groups ? 0 : 1);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        ++n_launches;
    }
    return cudaSuccess;
}

}  // namespace pcgrl
