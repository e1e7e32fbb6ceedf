// extern "C" surface of libpcgrl_sm100.so (see include/pcgrl_b200.h for the contract).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <string>
#include <vector>

#include "pcgrl_device.cuh"

namespace pcgrl {
cudaError_t launch_bitboard(const KParams& p, int problem, cudaStream_t s, bool& supported);
cudaError_t launch_bigboard(const KParams& p, int problem, cudaStream_t s, bool& supported);
cudaError_t launch_bitboard_split(const KParams& p, int problem, cudaStream_t s, int incremental, bool& supported,
                                  int& n_launches);
cudaError_t launch_bitboard_lanegroup(const KParams& p, int problem, cudaStream_t s, bool& supported);
int bitboard_cache_stride(int problem, int ndim, int d0, int d1, int rep, int action_kind);
int split_prog_search_warps(int64_t n);
bool split_prog_supported(const KParams& p, int problem);
cudaError_t launch_maze3d(const KParams& p, cudaStream_t s, bool& supported);
cudaError_t launch_maze3d_holey(const KParams& p, int problem, cudaStream_t s, bool& supported);
cudaError_t launch_sokoban(const KParams& p, cudaStream_t s, bool& supported);
cudaError_t launch_smb(const KParams& p, cudaStream_t s, bool& supported, int& n_launches);
int64_t sokoban_scratch_bytes();
int64_t smb_scratch_bytes(int64_t n_envs);
int64_t maze3d_scratch_bytes();
cudaError_t launch_observe(const pcgrl_config& cfg, const pcgrl_state& st, const pcgrl_obs_args& o, cudaStream_t s);
cudaError_t launch_update(const KParams& p, cudaStream_t s);

// split step path: up to WL_CHUNKS host-pipeline chunks, one 16-int work-list header each at the front of
// pcgrl_state.worklist
constexpr int WL_CHUNKS = 64, WL_HDR_INTS = 16 * WL_CHUNKS;

static thread_local std::string g_err;
static std::atomic<int64_t> g_launches{0};

static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
static int cuda_fail(cudaError_t e, const char* what) {
    return fail(PCGRL_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

static int cells_of(const pcgrl_config* c) { return c->dims[0] * c->dims[1] * (c->ndim == 3 ? c->dims[2] : 1); }

static int check(const pcgrl_config* c) {
    if (!c) return fail(PCGRL_E_ARG, "config is NULL");
    if (c->abi_version != PCGRL_ABI_VERSION) return fail(PCGRL_E_ARG, "abi_version mismatch");
    if (c->ndim != 2 && c->ndim != 3) return fail(PCGRL_E_ARG, "ndim must be 2 or 3");
    for (int i = 0; i < c->ndim; ++i)
        if (c->dims[i] < 1) return fail(PCGRL_E_ARG, "dims must be >= 1");
    if (c->n_tiles < 1 || c->n_tiles > PCGRL_MAX_TILES) return fail(PCGRL_E_ARG, "n_tiles out of range");
    if (c->n_stats < 1 || c->n_stats > PCGRL_MAX_STATS) return fail(PCGRL_E_ARG, "n_stats out of range");
    if (c->representation < PCGRL_REP_NARROW || c->representation > PCGRL_REP_CELLULAR)
        return fail(PCGRL_E_ARG, "unknown representation");
    const int cells = cells_of(c);
    if (c->row_stride < cells || c->row_stride % 16) return fail(PCGRL_E_ARG, "row_stride must be >= cells and a multiple of 16");
    static const int k_of[] = {2, 7, 7, 9, 3, 3, 2, 5, 6};
    if (c->problem < 0 || c->problem > PCGRL_PROB_MINECRAFT_3D_DUNGEON_HOLEY) return fail(PCGRL_E_ARG, "unknown problem");
    if ((c->problem == PCGRL_PROB_MINECRAFT_3D_HOLEY_MAZE || c->problem == PCGRL_PROB_MINECRAFT_3D_DUNGEON_HOLEY) && c->ndim != 3)
        return fail(PCGRL_E_ARG, "the minecraft holey problems are 3D");
    if (c->hole_mode < PCGRL_HOLES_GIVEN || c->hole_mode > PCGRL_HOLES_RANDOM) return fail(PCGRL_E_ARG, "unknown hole_mode");
    if (c->problem == PCGRL_PROB_BINARY_HOLEY && c->ndim != 2) return fail(PCGRL_E_ARG, "binary_holey is a 2D problem");
    if (c->n_stats != k_of[c->problem]) return fail(PCGRL_E_ARG, "n_stats does not match the problem");
    const int r = c->representation, a = c->action_kind;
    const bool ok = ((r == PCGRL_REP_NARROW || r == PCGRL_REP_TURTLE) && a == PCGRL_ACT_INT32) ||
                    (r == PCGRL_REP_NARROW && a == PCGRL_ACT_PATCH) ||
                    (r == PCGRL_REP_WIDE && (a == PCGRL_ACT_WIDE_COORDS || a == PCGRL_ACT_WIDE_FLAT)) ||
                    (r == PCGRL_REP_CELLULAR && (a == PCGRL_ACT_CA_TILES || a == PCGRL_ACT_CA_LOGITS));
    if (!ok) return fail(PCGRL_E_ARG, "action_kind does not fit the representation");
    if (a == PCGRL_ACT_WIDE_FLAT && (c->act_h < 1 || c->act_w < 1)) return fail(PCGRL_E_ARG, "act_h/act_w required");
    if (a == PCGRL_ACT_PATCH) {
        for (int i = 0; i < 3; ++i) {
            const int dim = i < c->ndim ? c->dims[i] : 1;
            if (c->act_window[i] < 1 || c->act_window[i] > dim)
                return fail(PCGRL_E_ARG, "act_window must be within [1, dim] on every axis (1 on unused axes)");
        }
    } else if (c->act_window[0] > 1 || c->act_window[1] > 1 || c->act_window[2] > 1) {
        return fail(PCGRL_E_ARG, "act_window needs action_kind PCGRL_ACT_PATCH (narrow representation)");
    }
    if (c->static_prob < 0.f || c->static_prob > 1.f || c->n_static_walls < 0)
        return fail(PCGRL_E_ARG, "static_prob must be in [0,1] and n_static_walls >= 0");
    if (c->n_static_walls > 0 && (c->wall_tile < 0 || c->wall_tile >= c->n_tiles))
        return fail(PCGRL_E_ARG, "wall_tile out of range");
    if (c->reward_mode != PCGRL_REWARD_CONTROL && c->reward_mode != PCGRL_REWARD_RANGE)
        return fail(PCGRL_E_ARG, "unknown reward_mode");
    const int ab = c->action_elem_bytes;
    if (ab != 0 && ab != 1 && ab != 2 && ab != 4) return fail(PCGRL_E_ARG, "action_elem_bytes must be 0, 1, 2 or 4");
    if ((ab == 1 || ab == 2) && a != PCGRL_ACT_INT32 && a != PCGRL_ACT_WIDE_FLAT)
        return fail(PCGRL_E_ARG, "narrow action elements only apply to scalar actions (PCGRL_ACT_INT32 / PCGRL_ACT_WIDE_FLAT)");
    if (ab == 1 || ab == 2) {   // every legal action must be representable
        const int64_t n_act = a == PCGRL_ACT_WIDE_FLAT ? (int64_t)c->act_h * c->act_w * c->n_tiles
                            : r == PCGRL_REP_TURTLE ? 4 + c->n_tiles : c->n_tiles;
        if (n_act > (ab == 1 ? 256 : 65536)) return fail(PCGRL_E_ARG, "action_elem_bytes too small for the action space");
    }
    const int sb = c->record_stat_bytes;
    if (sb != 0 && sb != 1 && sb != 2 && sb != 4) return fail(PCGRL_E_ARG, "record_stat_bytes must be 0, 1, 2 or 4");
    return 0;
}
// minecraft_2D_maze runs the binary kernels: same stats, its passable tile "AIR" is code 0 like binary's "empty"
static int kernel_problem(int problem) { return problem == PCGRL_PROB_MINECRAFT_2D_MAZE ? PCGRL_PROB_BINARY : problem; }
static bool is_bitboard(const pcgrl_config* c) {
    const int k = kernel_problem(c->problem);
    return k == PCGRL_PROB_BINARY || k == PCGRL_PROB_ZELDA || k == PCGRL_PROB_BINARY_HOLEY;
}
static int cache_stride(const pcgrl_config* c) {
    return bitboard_cache_stride(kernel_problem(c->problem), c->ndim, c->dims[0], c->dims[1], c->representation,
                                 c->action_kind);
}
// PCGRL_STEP_PATH = fused | split | inc | incfused | lg (default by shard size, step_path()): which of the equivalent step paths pcgrl_step
// takes when the caller supplied the buffers for all of them (A/B runs and the path-equivalence tests)
static int path_of(const char* e, int dflt) {
    if (!e) return dflt;
    return !strcmp(e, "fused") ? 0 : !strcmp(e, "split") ? 1 : !strcmp(e, "inc") ? 2 : !strcmp(e, "incfused") ? 3
         : !strcmp(e, "lg") ? 4 : dflt;
}
// Measured on B200, binary 16x16, ms per step of a shard of 64 Ki / 256 Ki / 512 Ki / 1 Mi envs:
//   fused 0.066 / 0.131 / 0.220 / 0.385   inc (3 launches) 0.063 / 0.114 / 0.175 / 0.304   incfused 0.058 / 0.122 / 0.203 / 0.367
// so a plain pcgrl_step takes the one-launch incremental kernel for small shards and the three-launch one above.
// The lane-group kernel (step_lanegroup.cu, path 4 "lg"; kernel times, profiles/r02_lanegroup_by_size.txt): 1 Ki / 4 Ki / 16 Ki
// envs 24.9 / 27.1 / 31.5 us against 30.8 / 32.6 / 33.7 us for incfused, 64 Ki 67.5 / 58.0 -- it takes the shards below 24 Ki envs
// (RLlib-scale batches).
// With its grid sized so that every CTA works and warps take two update rounds (step_split.cu, launch_split) the
// one-launch kernel holds up to ~256 Ki envs (profiles/r02_step_inc_rounds.txt, kernel ms incfused / inc: 160 Ki 0.086 / 0.105,
// 256 Ki 0.112-0.125 / 0.116, 384 Ki 0.166 / 0.143, 512 Ki 0.209 / 0.177): the three-launch path takes over at 224 Ki.
// zelda's searches are short (7x11 maps, three small BFS): the one-launch fused kernel beats the three-launch split path
// at every size (profiles/r02_zelda_paths.txt, kernel ms fused / split: 64 Ki envs 0.037 / 0.041, 256 Ki 0.058 / 0.075,
// 1 Mi 0.175 / 0.201), so zelda only takes the split path when PCGRL_STEP_PATH asks for it.
// The problems without a search cache (binary_holey, binary maps of 17..32 rows) run the from-scratch machines either
// way: fused below 128 Ki envs, the split path (full warps from a global list) above (profiles/r02_zelda_paths.txt:
// binary 24x24 64 Ki envs 0.207 / 0.227 ms fused / split, 512 Ki 1.019 / 0.943; binary_holey 64 Ki 0.087 / 0.086, 1 Mi 0.820 / 0.580).
static int step_path(int64_t n_envs, int problem, bool has_cache) {
    const int dflt = problem == PCGRL_PROB_ZELDA ? 0
                   : !has_cache ? (n_envs < (128 << 10) ? 0 : 1)
                   : n_envs < (24 << 10) ? 4 : n_envs < (224 << 10) ? 3 : 2;
    return path_of(getenv("PCGRL_STEP_PATH"), dflt);
}
// Chunks of the host pipeline run on different streams.  With the search kernel of the three-launch incremental
// path limited to 3 CTAs per SM (PCGRL_INC_CTAS_PER_SM_HOST) the memory-bound update / output kernels of the
// neighbouring chunks run NEXT TO it: e2e 2.60e9 env-steps/s at 4 chunks, against 2.24e9 with the fused kernel and
// 2.11e9 when the search holds every SM for itself (8 CTAs per SM); shards without a search cache keep the fused kernel
static int host_chunk_path(bool has_cache) { return has_cache ? path_of(getenv("PCGRL_HOST_PATH"), 2) : 0; }
static int action_elem(const pcgrl_config* c) { return c->action_elem_bytes ? c->action_elem_bytes : 4; }
static int record_stride(const pcgrl_config* c) {
    return c->record_stat_bytes ? (4 + c->n_stats * c->record_stat_bytes + 2 + 3) / 4 * 4 : 0;
}

static void fill(KParams& p, const pcgrl_config* c, const pcgrl_state* st) {
    std::memset(&p, 0, sizeof(p));
    p.rep = c->representation;
    p.action_kind = c->action_kind;
    p.ndim = c->ndim;
    p.d0 = c->dims[0];
    p.d1 = c->dims[1];
    p.d2 = c->ndim == 3 ? c->dims[2] : 1;
    p.cells = cells_of(c);
    p.row_stride = c->row_stride;
    p.n_tiles = c->n_tiles;
    p.n_stats = c->n_stats;
    p.max_iterations = c->max_iterations;
    p.max_changes = c->max_changes;
    p.act_h = c->act_h;
    p.act_w = c->act_w;
    p.targets_per_env = c->targets_per_env;
    p.init_random_probs = c->init_random_probs;
    p.reward_mode = c->reward_mode;
    const bool patch = c->action_kind == PCGRL_ACT_PATCH;
    p.aw0 = patch ? c->act_window[0] : 1;
    p.aw1 = patch ? c->act_window[1] : 1;
    p.aw2 = patch && c->ndim == 3 ? c->act_window[2] : 1;
    p.static_prob = c->static_prob;
    p.n_static_walls = c->n_static_walls;
    p.wall_tile = c->wall_tile;
    p.static_eval_mode = c->static_eval_mode;
    p.hole_mode = c->hole_mode;
    p.act_bytes = action_elem(c);
    p.rec_sb = c->record_stat_bytes;
    p.rec_stride = record_stride(c);
    double tot = 0;
    for (int t = 0; t < c->n_tiles; ++t) tot += c->init_probs[t] > 0 ? c->init_probs[t] : 0;
    double run = 0;
    for (int t = 0; t < c->n_tiles; ++t) {
        run += (c->init_probs[t] > 0 ? c->init_probs[t] : 0) / (tot > 0 ? tot : 1);
        p.init_cdf[t] = (float)run;
    }
    for (int k = 0; k < PCGRL_MAX_STATS; ++k) p.weights[k] = c->weights[k];
    if (st) {
        p.n_envs = st->n_envs;
        p.env_offset = st->env_offset;
        p.grids = st->grids;
        p.pos = st->pos;
        p.n_step = st->n_step;
        p.iteration = st->iteration;
        p.changes = st->changes;
        p.stats = st->stats;
        p.targets = st->targets;
        p.reward = st->reward;
        p.done = st->done;
        p.changed = st->changed;
        p.status = st->status;
        p.scratch = st->scratch;
        p.static_mask = st->static_mask;
        p.holes = st->holes;
        p.records = p.rec_sb ? st->records : nullptr;
        // split path: headers of up to WL_CHUNKS pipeline chunks at the front (16 ints each), bodies behind them
        p.wl_hdr = st->worklist;
        p.worklist = st->worklist ? st->worklist + WL_HDR_INTS : nullptr;
        p.cache_stride = cache_stride(c);
        p.cache = p.cache_stride && st->worklist ? st->cache : nullptr;
    }
}

static bool is_holey3d(const pcgrl_config* c) {
    return c->problem == PCGRL_PROB_MINECRAFT_3D_HOLEY_MAZE || c->problem == PCGRL_PROB_MINECRAFT_3D_DUNGEON_HOLEY;
}
static bool is_holey(const pcgrl_config* c) { return c->problem == PCGRL_PROB_BINARY_HOLEY || is_holey3d(c); }
static int hole_ints(const pcgrl_config* c) { return is_holey3d(c) ? 6 : 4; }

static int check_state(const pcgrl_state* st) {
    if (!st) return fail(PCGRL_E_ARG, "state is NULL");
    if (st->n_envs < 0) return fail(PCGRL_E_ARG, "n_envs < 0");
    if (!st->grids || !st->pos || !st->n_step || !st->iteration || !st->changes || !st->stats || !st->targets ||
        !st->reward || !st->done)
        return fail(PCGRL_E_ARG, "a required state pointer is NULL");
    return 0;
}

static int run(const KParams& p, int cfg_problem, void* stream, int force_path = -1) {
    const int problem = kernel_problem(cfg_problem);
    bool supported = false;
    int multi = 0;
    cudaError_t e;
    if (problem == PCGRL_PROB_MINECRAFT_3D_MAZE)
        e = launch_maze3d(p, (cudaStream_t)stream, supported);
    else if (problem == PCGRL_PROB_MINECRAFT_3D_HOLEY_MAZE || problem == PCGRL_PROB_MINECRAFT_3D_DUNGEON_HOLEY)
        e = launch_maze3d_holey(p, problem, (cudaStream_t)stream, supported);
    else if (problem == PCGRL_PROB_SOKOBAN)
        e = launch_sokoban(p, (cudaStream_t)stream, supported);
    else if (problem == PCGRL_PROB_SMB)
        e = launch_smb(p, (cudaStream_t)stream, supported, multi);   // map statistics + lane-group playthroughs + fallback
    else {
        int path = force_path >= 0 ? force_path : step_path(p.n_envs, problem, p.cache != nullptr);
        if (p.mode == MODE_STEP && path == 4) {   // lane groups (step_lanegroup.cu): small binary shards with a search cache
            if (p.cache) {
                e = launch_bitboard_lanegroup(p, problem, (cudaStream_t)stream, supported);
                if (supported) {
                    if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
                    g_launches.fetch_add(1, std::memory_order_relaxed);
                    return 0;
                }
            }
            path = 3;
        }
        if (p.mode == MODE_STEP && p.worklist && path > 0) {
            int n_launches = 0;
            e = launch_bitboard_split(p, problem, (cudaStream_t)stream, path - 1, supported, n_launches);
            if (supported) {
                if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
                g_launches.fetch_add(n_launches, std::memory_order_relaxed);
                return 0;
            }
        }
        if (p.split_phase != 0) return fail(PCGRL_E_UNSUPPORTED, "progressive host pipeline: config has no incremental split path");
        e = launch_bitboard(p, problem, (cudaStream_t)stream, supported);
        // maps beyond 32x32 (binary_bigger / zelda_bigger are 64x64): warp-per-grid boards
        if (!supported) e = launch_bigboard(p, problem, (cudaStream_t)stream, supported);
    }
    if (!supported)
        return fail(PCGRL_E_UNSUPPORTED, "no kernel for this problem / map shape yet (or scratch is NULL although "
                                         "pcgrl_scratch_bytes() > 0)");
    if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
    // sokoban: step kernel + BFS jobs + A* jobs + combine (step_sokoban.cu)
    g_launches.fetch_add(problem == PCGRL_PROB_SOKOBAN ? 4 : (multi ? multi : 1), std::memory_order_relaxed);
    return 0;
}
// Chunked, stream-pipelined host step: the shard is cut into chunks of whole CTA tiles; every chunk's action upload
// is queued on the upload stream, its step kernels on compute stream c % n_compute, its result download on the
// download stream (events in between), so uploads, kernels and downloads of different chunks overlap (two copy
// engines + the SMs) and a chunk never waits for another chunk's download.
// Only for kernels that keep no cross-launch device state (scratch == 0, i.e. not the persistent solvers).
constexpr int PIPE_COMPUTE_MAX = 6;             // streams the chunks' kernels rotate over: n_compute of them (PCGRL_HOST_STREAMS)
constexpr int PIPE_STREAMS = PIPE_COMPUTE_MAX + 2;  // + one upload stream and one download stream (the last two)
static int pipe_compute() {
    static const int v = getenv("PCGRL_HOST_STREAMS") ? std::min(std::max(atoi(getenv("PCGRL_HOST_STREAMS")), 1), PIPE_COMPUTE_MAX) : 3;
    return v;
}
struct HostGraphKey {            // everything the queued operations depend on (compared bytewise)
    pcgrl_config cfg;
    pcgrl_state st;
    void* actions_dev;
    int64_t action_bytes;
    int64_t has_host_actions;
    void *reward_host, *done_host, *stats_host, *records_host;
    int32_t chunks, chunk_path;
};
struct HostGraph {
    struct Upload {
        cudaGraphNode_t node;
        void* dst;
        int64_t off;
        size_t bytes;
    };
    HostGraphKey key;
    cudaGraph_t graph = nullptr;     // kept alive: the upload nodes updated in `exec` are named by their handles in it
    cudaGraphExec_t exec = nullptr;
    std::vector<Upload> h2d;
    const void* last_src = nullptr;
    int64_t launches = 0;
};
struct HostPipe {
    static constexpr int MAX_GRAPHS = 8;
    bool ready = false, graph_broken = false;
    cudaStream_t s[PIPE_STREAMS];
    cudaEvent_t fork, join[PIPE_STREAMS];
    cudaEvent_t up_ev[WL_CHUNKS], k_ev[WL_CHUNKS];   // chunk c's actions are on the device / its kernels are done
    HostGraph graphs[MAX_GRAPHS];
    unsigned next_graph = 0;
};
static thread_local HostPipe g_pipe[16];

// smallest shard the progressive host pipeline takes (read per call: the tests lower it)
static int64_t prog_min_envs() {
    const char* e = getenv("PCGRL_HOST_PROG_MIN");
    return e ? atoll(e) : (int64_t)1 << 18;
}
static int host_chunks(const pcgrl_config* cfg, int64_t n, bool packed) {
    (void)packed;
    if (!is_bitboard(cfg) || cfg->dims[0] > 32 || cfg->dims[1] > 32) return 1;
    if (const char* e = getenv("PCGRL_HOST_CHUNKS")) {
        const int v = atoi(e);
        if (v >= 1) return (int)std::min<int64_t>(std::min(v, WL_CHUNKS), std::max<int64_t>(1, n / 256));
    }
    // measured on B200 (binary 16x16, e2e env-steps/s): 64 Ki envs 1 chunk best (2 / 4 chunks: 3.3 / 2.4e8); 256 Ki
    // 1 / 2 / 4 chunks -> 8.5 / 9.1 / 7.1e8; 512 Ki -> 1.07 / 1.26 / 1.09e9; 1 Mi 2 / 4 / 8 -> 1.77 / 2.0 / 1.77e9.
    // Every chunk costs ~18 us of queue operations, so small shards take fewer.
    // With the copies on their own streams (profiles/r02_e2e_chunks_by_size.txt): 128 Ki 1 / 2 / 3 / 4 chunks -> 8.9 / 9.2 /
    // 8.7 / 8.5e8; 256 Ki -> 1.40 / 1.44 / 1.35 / 1.30e9; 512 Ki -> 1.82 / 1.84 / 2.05 / 2.09e9; 1 Mi 4 / 6 / 8 -> 2.75 / 2.73 / 2.54e9.
    if (n < (1 << 17)) return 1;
    if (n < (1 << 19)) return 2;
    return 4;
}
}  // namespace pcgrl

using namespace pcgrl;

extern "C" {

int32_t pcgrl_abi_version(void) { return PCGRL_ABI_VERSION; }
const char* pcgrl_last_error(void) { return g_err.c_str(); }
int64_t pcgrl_launch_count(void) { return g_launches.load(); }

int32_t pcgrl_config_check(pcgrl_config* cfg) {
    if (!cfg) return fail(PCGRL_E_ARG, "config is NULL");
    if (cfg->row_stride == 0 && (cfg->ndim == 2 || cfg->ndim == 3)) cfg->row_stride = (cells_of(cfg) + 15) / 16 * 16;
    return check(cfg);
}

int64_t pcgrl_scratch_bytes(const pcgrl_config* cfg, int64_t n_envs) {
    if (check(cfg)) return -1;
    // node pools / heaps / hash tables of the solver problems: one slice per resident search warp
    if (cfg->problem == PCGRL_PROB_SOKOBAN) return sokoban_scratch_bytes();
    if (cfg->problem == PCGRL_PROB_SMB) return smb_scratch_bytes(n_envs);   // + the per-env length history
    if (cfg->problem == PCGRL_PROB_MINECRAFT_3D_MAZE || is_holey3d(cfg)) return maze3d_scratch_bytes();   // jump counts, parents
    return 0;  // binary / zelda keep all search state in registers / shared memory
}

int64_t pcgrl_step_bytes(const pcgrl_config* c) {
    if (check(c)) return -1;
    const int64_t G = cells_of(c), K = c->n_stats;
    int64_t A = action_elem(c);
    if (c->action_kind == PCGRL_ACT_WIDE_COORDS) A = 4 * (c->ndim + 1);
    if (c->action_kind == PCGRL_ACT_CA_TILES) A = G;
    if (c->action_kind == PCGRL_ACT_PATCH)
        A = 4 * (int64_t)c->act_window[0] * c->act_window[1] * (c->ndim == 3 ? c->act_window[2] : 1);
    if (c->action_kind == PCGRL_ACT_CA_LOGITS) A = 4 * (int64_t)c->n_tiles * G;
    return 2 * G + A + 8 * K + 5 + (c->targets_per_env ? 16 * K : 0);
}

int64_t pcgrl_worklist_ints(const pcgrl_config* cfg, int64_t n_envs) {
    if (check(cfg) || n_envs < 0) return -1;
    if (!is_bitboard(cfg) || cfg->representation == PCGRL_REP_CELLULAR || cfg->ndim != 2) return 0;
    if (cfg->dims[0] > 32 || cfg->dims[1] > 32) return 0;   // warp-per-grid boards (step_bigboard.cu): fused only
    // header + (env, cell) + new stats per env, plus one header per host-pipeline chunk (up to 64)
    return (2 + (int64_t)cfg->n_stats) * n_envs + WL_HDR_INTS;
}

int32_t pcgrl_cache_stride(const pcgrl_config* cfg) {
    if (check(cfg)) return -1;
    return cache_stride(cfg);
}

int32_t pcgrl_record_stride(const pcgrl_config* cfg) {
    if (check(cfg)) return -1;
    return record_stride(cfg);
}

// One step launch over `st`.  wl_chunk / wl_off place this launch's work list inside the PARENT shard's
// pcgrl_state.worklist (host pipeline: st is a sub-range starting wl_off envs into the shard and `wl_base` is the
// parent's buffer); a plain pcgrl_step is chunk 0 at offset 0 of its own buffer.
static int32_t step_launch(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions, void* stream,
                           int32_t* wl_base, int wl_chunk, int64_t wl_off, int force_path = -1, int phase = 0,
                           int ml_lists = 0, int64_t ml_per = 0, int ml_target = 0) {
    int r = check(cfg);
    if (r) return r;
    if ((r = check_state(st))) return r;
    if (!actions) return fail(PCGRL_E_ARG, "actions is NULL");
    if (is_holey(cfg) && !st->holes) return fail(PCGRL_E_ARG, "a holey problem needs pcgrl_state.holes");
    KParams p;
    fill(p, cfg, st);
    if (wl_base) {
        p.wl_hdr = wl_base + 16 * wl_chunk;
        p.worklist = wl_base + WL_HDR_INTS + (2 + (int64_t)cfg->n_stats) * wl_off;
    }
    p.mode = MODE_STEP;
    p.actions = actions;
    p.host_chunk = force_path >= 0;
    p.split_phase = phase;
    p.ml_lists = ml_lists;
    p.ml_per = ml_per;
    p.ml_target = ml_target;
    return run(p, cfg->problem, stream, force_path);
}

int32_t pcgrl_step(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions, void* stream) {
    return step_launch(cfg, st, actions, stream, st ? st->worklist : nullptr, 0, 0);
}

int32_t pcgrl_update(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions, void* stream) {
    int r = check(cfg);
    if (r) return r;
    // only what the update touches: a holey problem's holes, the counters and the stats are not read
    if (!st) return fail(PCGRL_E_ARG, "state is NULL");
    if (st->n_envs < 0) return fail(PCGRL_E_ARG, "n_envs < 0");
    if (!st->grids || !st->pos || !st->n_step || !st->changed)
        return fail(PCGRL_E_ARG, "pcgrl_update needs grids, pos, n_step and changed");
    if (!actions) return fail(PCGRL_E_ARG, "actions is NULL");
    KParams p;
    fill(p, cfg, st);
    p.mode = MODE_STEP;
    p.actions = actions;
    const cudaError_t e = launch_update(p, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "update launch");
    if (st->n_envs > 0) g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

int32_t pcgrl_reset(const pcgrl_config* cfg, const pcgrl_state* st, const uint8_t* mask, const int8_t* src_grids,
                    const int32_t* src_pos, uint64_t seed, uint64_t epoch, void* stream) {
    int r = check(cfg);
    if (r) return r;
    if ((r = check_state(st))) return r;
    if (is_holey(cfg) && !st->holes) return fail(PCGRL_E_ARG, "a holey problem needs pcgrl_state.holes");
    KParams p;
    fill(p, cfg, st);
    if (!is_holey(cfg)) p.holes = nullptr;
    p.mode = MODE_RESET;
    p.mask = mask;
    p.src_grids = src_grids;
    p.src_pos = src_pos;
    p.seed = seed;
    p.epoch = epoch;
    return run(p, cfg->problem, stream);
}

int32_t pcgrl_stats(const pcgrl_config* cfg, const int8_t* grids, int32_t* stats, int64_t n, void* scratch,
                    void* stream) {
    int r = check(cfg);
    if (r) return r;
    if (!grids || !stats || n < 0) return fail(PCGRL_E_ARG, "bad grids/stats/n");
    if (is_holey(cfg)) return fail(PCGRL_E_ARG, "a holey problem needs pcgrl_stats_holey (entrance / exit per grid)");
    KParams p;
    fill(p, cfg, nullptr);
    p.mode = MODE_STATS;
    p.n_envs = n;
    p.stats_grids = grids;
    p.stats_out = stats;
    p.scratch = scratch;
    return run(p, cfg->problem, stream);
}

int32_t pcgrl_stats_holey(const pcgrl_config* cfg, const int8_t* grids, const int32_t* holes, int32_t* stats,
                          int64_t n, void* scratch, void* stream) {
    int r = check(cfg);
    if (r) return r;
    if (!grids || !stats || !holes || n < 0) return fail(PCGRL_E_ARG, "bad grids/holes/stats/n");
    if (!is_holey(cfg)) return fail(PCGRL_E_ARG, "pcgrl_stats_holey needs a holey problem");
    KParams p;
    fill(p, cfg, nullptr);
    p.mode = MODE_STATS;
    p.n_envs = n;
    p.stats_grids = grids;
    p.stats_out = stats;
    p.scratch = scratch;
    p.holes = const_cast<int32_t*>(holes);
    return run(p, cfg->problem, stream);
}

int32_t pcgrl_observe(const pcgrl_config* cfg, const pcgrl_state* st, const pcgrl_obs_args* obs, void* stream) {
    int r = check(cfg);
    if (r) return r;
    if (!st || !st->grids || !st->pos || !obs || !obs->out) return fail(PCGRL_E_ARG, "bad observe arguments");
    if (obs->n_ctrl < 0 || obs->n_ctrl > PCGRL_MAX_STATS) return fail(PCGRL_E_ARG, "n_ctrl out of range");
    if (obs->n_ctrl > 0 && (!st->stats || !st->targets)) return fail(PCGRL_E_ARG, "control channels need stats/targets");
    cudaError_t e = launch_observe(*cfg, *st, *obs, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "observe launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

// Shared body of pcgrl_step_host / pcgrl_step_host_packed: with records_host the only download is the packed
// record range of each chunk (one copy); otherwise reward / done / stats are copied separately.
static int32_t step_host_impl(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions_host, void* actions_dev,
                              int64_t action_bytes, float* reward_host, uint8_t* done_host, int32_t* stats_host,
                              uint8_t* records_host, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e;
    int r = check(cfg);
    if (r) return r;
    if ((r = check_state(st))) return r;
    if (actions_host && (!actions_dev || action_bytes < 0)) return fail(PCGRL_E_ARG, "actions_dev / action_bytes");
    if (!actions_dev) return fail(PCGRL_E_ARG, "actions_dev is NULL");
    const int64_t rs = record_stride(cfg);
    if (records_host && (!st->records || rs == 0))
        return fail(PCGRL_E_ARG, "packed host step needs cfg.record_stat_bytes and pcgrl_state.records");
    const int64_t n = st->n_envs;
    const int K = cfg->n_stats;
    int chunks = (n > 0 && (!actions_host || action_bytes % n == 0)) ? host_chunks(cfg, n, records_host != nullptr) : 1;
    if (chunks <= 1) {
        if (actions_host &&
            (e = cudaMemcpyAsync(actions_dev, actions_host, (size_t)action_bytes, cudaMemcpyHostToDevice, s)) != cudaSuccess)
            return cuda_fail(e, "H2D actions");
        if ((r = pcgrl_step(cfg, st, actions_dev, stream))) return r;
        if (records_host && (e = cudaMemcpyAsync(records_host, st->records, (size_t)(n * rs), cudaMemcpyDeviceToHost, s)) != cudaSuccess)
            return cuda_fail(e, "D2H records");
        if (reward_host && (e = cudaMemcpyAsync(reward_host, st->reward, n * sizeof(float), cudaMemcpyDeviceToHost, s)) != cudaSuccess)
            return cuda_fail(e, "D2H reward");
        if (done_host && (e = cudaMemcpyAsync(done_host, st->done, n, cudaMemcpyDeviceToHost, s)) != cudaSuccess)
            return cuda_fail(e, "D2H done");
        if (stats_host && (e = cudaMemcpyAsync(stats_host, st->stats, n * K * sizeof(int32_t), cudaMemcpyDeviceToHost, s)) != cudaSuccess)
            return cuda_fail(e, "D2H stats");
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return cuda_fail(e, "stream sync");
        return 0;
    }

    int dev = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
    if (dev < 0 || dev >= 16) return fail(PCGRL_E_ARG, "device index out of range for the host pipeline");
    HostPipe& hp = g_pipe[dev];
    if (!hp.ready) {
        for (int i = 0; i < PIPE_STREAMS; ++i) {
            if ((e = cudaStreamCreateWithFlags(&hp.s[i], cudaStreamNonBlocking)) != cudaSuccess) return cuda_fail(e, "stream create");
            if ((e = cudaEventCreateWithFlags(&hp.join[i], cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(e, "event create");
        }
        if ((e = cudaEventCreateWithFlags(&hp.fork, cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(e, "event create");
        for (int i = 0; i < WL_CHUNKS; ++i)
            if ((e = cudaEventCreateWithFlags(&hp.up_ev[i], cudaEventDisableTiming)) != cudaSuccess ||
                (e = cudaEventCreateWithFlags(&hp.k_ev[i], cudaEventDisableTiming)) != cudaSuccess)
                return cuda_fail(e, "event create");
        hp.ready = true;
    }
    const int chunk_path = host_chunk_path(st->worklist && st->cache && cache_stride(cfg) > 0);
    // Progressive pipeline (binary maps <= 16x16 with the incremental search, from 256 Ki envs): every chunk's update
    // kernel, then ONE search over all the chunks' lists in chunk order (k_split_stats_inc_multi), and per chunk a
    // wait kernel + output kernel + download that go as soon as the search has finished that chunk's list -- the
    // search keeps the SIMT fill of the whole-shard launch and the downloads hide behind it.  PCGRL_HOST_PROG=0: the
    // chunk-per-stream pipeline below (three launches per chunk on rotating streams).
    const char* prog_env = getenv("PCGRL_HOST_PROG");
    const bool prog_on = prog_env && atoi(prog_env) != 0;
    bool prog = false;
    if (prog_on && chunk_path == 2 && n >= prog_min_envs() && cfg->n_stats == 2) {
        KParams probe;
        fill(probe, cfg, st);
        prog = split_prog_supported(probe, kernel_problem(cfg->problem));
    }
    if (prog && !getenv("PCGRL_HOST_CHUNKS")) chunks = n >= (1 << 19) ? 8 : 4;
    const int64_t per = ((n + chunks - 1) / chunks + 255) / 256 * 256;   // whole CTA tiles per chunk
    const int64_t a_env = actions_host ? action_bytes / n : 0;

    // PCGRL_HOST_TRACE=n: device timeline of n pipelined calls after 40 warm ones (events after every chunk's upload, kernels
    // and download, printed to stderr in microseconds from the fork) -- the stand-in for an nsys trace of the host leg.
    // Tracing queues the operations directly (no CUDA graph).
    static int trace_left = getenv("PCGRL_HOST_TRACE") ? atoi(getenv("PCGRL_HOST_TRACE")) : 0;
    static int trace_skip = 40;            // warm calls first (graph capture, clocks, pinned pages)
    static cudaEvent_t trace_ev[3 * WL_CHUNKS + 1];
    static bool trace_ready = false;
    cudaEvent_t* trace = nullptr;
    if (trace_left > 0 && trace_skip > 0) --trace_skip;
    else if (trace_left > 0) {
        if (!trace_ready) {
            for (auto& ev : trace_ev) cudaEventCreate(&ev);
            trace_ready = true;
        }
        trace = trace_ev;
    }
    // Queue every chunk: its upload on the upload stream, its kernels on compute stream c % PIPE_COMPUTE, its download
    // on the download stream, chained by events.  (With the copies on the compute stream itself, chunk c + 3 could not
    // start before chunk c's DOWNLOAD had finished -- the device trace, PCGRL_HOST_TRACE, showed the fourth chunk's
    // kernels starting 60 us after the first chunk's had ended.  PCGRL_HOST_SPLIT_COPIES=0 restores that order.)
    static const bool split_copies = !(getenv("PCGRL_HOST_SPLIT_COPIES") && atoi(getenv("PCGRL_HOST_SPLIT_COPIES")) == 0);
    auto enqueue_chunks = [&]() -> int {
        struct Chunk {
            int64_t off, m;
            char* a_dev;
            pcgrl_state sub;
        } ck[WL_CHUNKS];
        int n_ck = 0;
        for (int64_t off = 0; off < n; off += per, ++n_ck) {
            Chunk& q = ck[n_ck];
            const int64_t m = std::min(per, n - off);
            q.off = off;
            q.m = m;
            pcgrl_state& sub = q.sub;
            sub = *st;
            sub.n_envs = m;
            sub.env_offset = st->env_offset + off;
            sub.grids = st->grids + off * cfg->row_stride;
            sub.pos = st->pos + off * 3;
            sub.n_step = st->n_step + off;
            sub.iteration = st->iteration + off;
            sub.changes = st->changes + off;
            sub.stats = st->stats + off * K;
            sub.targets = st->targets + (cfg->targets_per_env ? off * K * 2 : 0);
            sub.reward = st->reward + off;
            sub.done = st->done + off;
            sub.changed = st->changed ? st->changed + off : nullptr;
            sub.static_mask = st->static_mask ? st->static_mask + off * cfg->row_stride : nullptr;
            sub.holes = st->holes ? st->holes + off * hole_ints(cfg) : nullptr;
            sub.records = st->records ? st->records + off * rs : nullptr;
            sub.cache = st->cache ? st->cache + off * cache_stride(cfg) : nullptr;
            int64_t a_stride = a_env;
            if (!actions_host) {   // actions already on the device: per-env stride from the action layout
                a_stride = cfg->action_kind == PCGRL_ACT_WIDE_COORDS ? 4 * (cfg->ndim + 1)
                         : cfg->action_kind == PCGRL_ACT_PATCH
                             ? 4 * (int64_t)cfg->act_window[0] * cfg->act_window[1] * (cfg->ndim == 3 ? cfg->act_window[2] : 1)
                         : cfg->action_kind == PCGRL_ACT_CA_TILES ? cfg->row_stride
                         : cfg->action_kind == PCGRL_ACT_CA_LOGITS ? 4 * (int64_t)cfg->n_tiles * cells_of(cfg) : action_elem(cfg);
            }
            q.a_dev = (char*)actions_dev + off * a_stride;
        }
        const int PIPE_COMPUTE = pipe_compute();
        cudaStream_t up = hp.s[PIPE_COMPUTE_MAX], down = hp.s[PIPE_COMPUTE_MAX + 1];
        if (prog) {
            cudaStream_t cs = hp.s[0], os = hp.s[1];
            const int target = split_prog_search_warps(n);
            if (target <= 0) return fail(PCGRL_E_CUDA, "progressive host pipeline: no SM count");
            for (int c = 0; c < n_ck && actions_host; ++c) {
                if ((e = cudaMemcpyAsync(ck[c].a_dev, (const char*)actions_host + ck[c].off * a_env, (size_t)(ck[c].m * a_env),
                                         cudaMemcpyHostToDevice, up)) != cudaSuccess)
                    return cuda_fail(e, "H2D actions");
                if ((e = cudaEventRecord(hp.up_ev[c], up)) != cudaSuccess) return cuda_fail(e, "event record");
                if (trace) cudaEventRecord(trace[3 * c + 0], up);
            }
            for (int c = 0; c < n_ck; ++c) {     // update kernels, chunk by chunk as the uploads land
                if (actions_host && (e = cudaStreamWaitEvent(cs, hp.up_ev[c], 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
                if (!actions_host && trace) cudaEventRecord(trace[3 * c + 0], cs);
                int rr = step_launch(cfg, &ck[c].sub, ck[c].a_dev, cs, st->worklist, c, ck[c].off, chunk_path, 1);
                if (rr) return rr;
            }
            // ONE search over every chunk's list; queued BEFORE the wait kernels so that none of them can sit in front
            // of it in a hardware queue
            int rr = step_launch(cfg, st, actions_dev, cs, st->worklist, 0, 0, chunk_path, 2, n_ck, per);
            if (rr) return rr;
            for (int c = 0; c < n_ck; ++c) {     // per chunk: wait for its list, output kernel, download
                const int64_t off = ck[c].off, m = ck[c].m;
                const pcgrl_state& sub = ck[c].sub;
                if ((rr = step_launch(cfg, &sub, ck[c].a_dev, os, st->worklist, c, off, chunk_path, 3, 0, 0, target))) return rr;
                if (trace) cudaEventRecord(trace[3 * c + 1], os);
                if ((e = cudaEventRecord(hp.k_ev[c], os)) != cudaSuccess) return cuda_fail(e, "event record");
                if ((e = cudaStreamWaitEvent(down, hp.k_ev[c], 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
                if (records_host && (e = cudaMemcpyAsync(records_host + off * rs, sub.records, (size_t)(m * rs), cudaMemcpyDeviceToHost, down)) != cudaSuccess)
                    return cuda_fail(e, "D2H records");
                if (reward_host && (e = cudaMemcpyAsync(reward_host + off, sub.reward, m * sizeof(float), cudaMemcpyDeviceToHost, down)) != cudaSuccess)
                    return cuda_fail(e, "D2H reward");
                if (done_host && (e = cudaMemcpyAsync(done_host + off, sub.done, m, cudaMemcpyDeviceToHost, down)) != cudaSuccess)
                    return cuda_fail(e, "D2H done");
                if (stats_host && (e = cudaMemcpyAsync(stats_host + off * K, sub.stats, m * K * sizeof(int32_t), cudaMemcpyDeviceToHost, down)) != cudaSuccess)
                    return cuda_fail(e, "D2H stats");
                if (trace) cudaEventRecord(trace[3 * c + 2], down);
            }
            return 0;
        }
        // every upload first: 1 B per env, on its own stream, long before the chunk's turn comes
        for (int c = 0; c < n_ck && actions_host; ++c) {
            cudaStream_t us = split_copies ? up : hp.s[c % PIPE_COMPUTE];
            if (!split_copies) continue;       // (old order: uploaded below, on the compute stream)
            if ((e = cudaMemcpyAsync(ck[c].a_dev, (const char*)actions_host + ck[c].off * a_env, (size_t)(ck[c].m * a_env),
                                     cudaMemcpyHostToDevice, us)) != cudaSuccess)
                return cuda_fail(e, "H2D actions");
            if ((e = cudaEventRecord(hp.up_ev[c], us)) != cudaSuccess) return cuda_fail(e, "event record");
            if (trace) cudaEventRecord(trace[3 * c + 0], us);
        }
        for (int c = 0; c < n_ck; ++c) {
            const int64_t off = ck[c].off, m = ck[c].m;
            const pcgrl_state& sub = ck[c].sub;
            cudaStream_t cs = hp.s[c % PIPE_COMPUTE];
            if (actions_host) {
                if (split_copies) {
                    if ((e = cudaStreamWaitEvent(cs, hp.up_ev[c], 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
                } else {
                    if ((e = cudaMemcpyAsync(ck[c].a_dev, (const char*)actions_host + off * a_env, (size_t)(m * a_env),
                                             cudaMemcpyHostToDevice, cs)) != cudaSuccess)
                        return cuda_fail(e, "H2D actions");
                    if (trace) cudaEventRecord(trace[3 * c + 0], cs);
                }
            } else if (trace) {
                cudaEventRecord(trace[3 * c + 0], cs);
            }
            // every chunk gets its own header and its own body range of the shard's work list
            int rr = step_launch(cfg, &sub, ck[c].a_dev, cs, st->worklist, c, off, chunk_path);
            if (rr) return rr;
            if (trace) cudaEventRecord(trace[3 * c + 1], cs);
            cudaStream_t ds = cs;
            if (split_copies) {
                if ((e = cudaEventRecord(hp.k_ev[c], cs)) != cudaSuccess) return cuda_fail(e, "event record");
                if ((e = cudaStreamWaitEvent(down, hp.k_ev[c], 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
                ds = down;
            }
            if (records_host && (e = cudaMemcpyAsync(records_host + off * rs, sub.records, (size_t)(m * rs), cudaMemcpyDeviceToHost, ds)) != cudaSuccess)
                return cuda_fail(e, "D2H records");
            if (reward_host && (e = cudaMemcpyAsync(reward_host + off, sub.reward, m * sizeof(float), cudaMemcpyDeviceToHost, ds)) != cudaSuccess)
                return cuda_fail(e, "D2H reward");
            if (done_host && (e = cudaMemcpyAsync(done_host + off, sub.done, m, cudaMemcpyDeviceToHost, ds)) != cudaSuccess)
                return cuda_fail(e, "D2H done");
            if (stats_host && (e = cudaMemcpyAsync(stats_host + off * K, sub.stats, m * K * sizeof(int32_t), cudaMemcpyDeviceToHost, ds)) != cudaSuccess)
                return cuda_fail(e, "D2H stats");
            if (trace) cudaEventRecord(trace[3 * c + 2], ds);
        }
        return 0;
    };

    // ---- CUDA graph of the whole pipeline -------------------------------------------------------------------------
    // A step of the host pipeline is ~25 queue operations (copies, launches, events over five streams) whose CPU cost sits
    // on the critical path of every step: the first kernel cannot start before its upload is queued, and the call
    // cannot return before the last event is.  The operations only depend on the pointers, so they are captured ONCE
    // (stream capture on helper stream 0, the others forked / joined by events inside the capture) and replayed
    // with one cudaGraphLaunch; only the source addresses of the uploads change from step to step
    // (cudaGraphExecMemcpyNodeSetParams1D).  PCGRL_HOST_GRAPH=0 queues the operations directly, as before.
    static const bool use_graph = !(getenv("PCGRL_HOST_GRAPH") && atoi(getenv("PCGRL_HOST_GRAPH")) == 0);
    // (the progressive pipeline is queued directly: only its first few operations -- uploads, update kernels, the search --
    // sit on the critical path, the rest is queued while the search runs)
    if (use_graph && !hp.graph_broken && !trace && !prog) {
        HostGraphKey key;
        std::memset(&key, 0, sizeof(key));
        key.cfg = *cfg;
        key.st = *st;
        key.actions_dev = actions_dev;
        key.action_bytes = action_bytes;
        key.has_host_actions = actions_host != nullptr;
        key.reward_host = reward_host;
        key.done_host = done_host;
        key.stats_host = stats_host;
        key.records_host = records_host;
        key.chunks = chunks;
        key.chunk_path = chunk_path;
        HostGraph* hg = nullptr;
        for (auto& g : hp.graphs)
            if (g.exec && !std::memcmp(&g.key, &key, sizeof(key))) hg = &g;
        if (!hg) {
            HostGraph& slot = hp.graphs[hp.next_graph++ % HostPipe::MAX_GRAPHS];
            if (slot.exec) cudaGraphExecDestroy(slot.exec);
            if (slot.graph) cudaGraphDestroy(slot.graph);
            slot.exec = nullptr;
            slot.graph = nullptr;
            slot.h2d.clear();
            cudaGraph_t graph = nullptr;
            bool ok = cudaStreamBeginCapture(hp.s[0], cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            if (ok) {
                ok = cudaEventRecord(hp.fork, hp.s[0]) == cudaSuccess;
                for (int i = 1; ok && i < PIPE_STREAMS; ++i) ok = cudaStreamWaitEvent(hp.s[i], hp.fork, 0) == cudaSuccess;
                const int64_t l0 = g_launches.load(std::memory_order_relaxed);
                const int rr = ok ? enqueue_chunks() : -1;
                slot.launches = g_launches.load(std::memory_order_relaxed) - l0;
                g_launches.fetch_sub(slot.launches, std::memory_order_relaxed);   // captured, not run: replays count them
                ok = ok && rr == 0;
                for (int i = 1; i < PIPE_STREAMS; ++i) {   // always join, so that the capture can end
                    const bool j1 = cudaEventRecord(hp.join[i], hp.s[i]) == cudaSuccess;
                    const bool j2 = cudaStreamWaitEvent(hp.s[0], hp.join[i], 0) == cudaSuccess;
                    ok = ok && j1 && j2;
                }
                ok = (cudaStreamEndCapture(hp.s[0], &graph) == cudaSuccess) && ok && graph;
            }
            if (ok) ok = cudaGraphInstantiate(&slot.exec, graph, 0) == cudaSuccess;
            if (ok && actions_host) {   // the upload nodes, by destination address = chunk
                size_t nn = 0;
                ok = cudaGraphGetNodes(graph, nullptr, &nn) == cudaSuccess;
                std::vector<cudaGraphNode_t> nodes(nn);
                if (ok && nn) ok = cudaGraphGetNodes(graph, nodes.data(), &nn) == cudaSuccess;
                for (size_t k = 0; ok && k < nn; ++k) {
                    cudaGraphNodeType ty;
                    if (cudaGraphNodeGetType(nodes[k], &ty) != cudaSuccess || ty != cudaGraphNodeTypeMemcpy) continue;
                    cudaMemcpy3DParms mp;
                    if (cudaGraphMemcpyNodeGetParams(nodes[k], &mp) != cudaSuccess) continue;
                    const char* dst = (const char*)mp.dstPtr.ptr;
                    if (dst < (const char*)actions_dev || dst >= (const char*)actions_dev + action_bytes) continue;
                    HostGraph::Upload u;
                    u.node = nodes[k];
                    u.dst = (void*)dst;
                    u.off = dst - (const char*)actions_dev;     // a_stride == a_env when the actions come from the host
                    u.bytes = mp.extent.width;
                    slot.h2d.push_back(u);
                }
                ok = ok && !slot.h2d.empty();
            }
            if (!ok) {
                if (graph) cudaGraphDestroy(graph);
                if (slot.exec) cudaGraphExecDestroy(slot.exec);
                slot.exec = nullptr;
                hp.graph_broken = true;     // e.g. a driver that cannot capture one of the operations: stay on the direct path
                cudaGetLastError();
            } else {
                slot.key = key;
                slot.graph = graph;
                slot.last_src = nullptr;
                hg = &slot;
            }
        }
        if (hg) {
            if (actions_host && hg->last_src != actions_host) {
                for (const auto& u : hg->h2d)
                    if ((e = cudaGraphExecMemcpyNodeSetParams1D(hg->exec, u.node, u.dst, (const char*)actions_host + u.off, u.bytes,
                                                                cudaMemcpyHostToDevice)) != cudaSuccess)
                        return cuda_fail(e, "graph upload update");
                hg->last_src = actions_host;
            }
            // after everything already queued on the caller's stream; the caller's stream continues after the graph
            if ((e = cudaEventRecord(hp.fork, s)) != cudaSuccess) return cuda_fail(e, "event record");
            if ((e = cudaStreamWaitEvent(hp.s[0], hp.fork, 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
            if ((e = cudaGraphLaunch(hg->exec, hp.s[0])) != cudaSuccess) return cuda_fail(e, "graph launch");
            if ((e = cudaEventRecord(hp.join[0], hp.s[0])) != cudaSuccess) return cuda_fail(e, "event record");
            if ((e = cudaStreamWaitEvent(s, hp.join[0], 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
            if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return cuda_fail(e, "stream sync");
            // the launches inside the graph are replayed, not re-issued: count them for pcgrl_launch_count
            g_launches.fetch_add(hg->launches, std::memory_order_relaxed);
            return 0;
        }
    }

    // ---- direct path: helper streams start after everything already queued on the caller's stream --------------------
    if (trace) cudaEventRecord(trace[3 * WL_CHUNKS], s);
    if ((e = cudaEventRecord(hp.fork, s)) != cudaSuccess) return cuda_fail(e, "event record");
    for (int i = 0; i < PIPE_STREAMS; ++i)
        if ((e = cudaStreamWaitEvent(hp.s[i], hp.fork, 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
    const auto t_host0 = std::chrono::steady_clock::now();
    if ((r = enqueue_chunks())) return r;
    const auto t_host1 = std::chrono::steady_clock::now();
    // join: later work on the caller's stream (auto-reset, observe) is ordered after every chunk
    for (int i = 0; i < PIPE_STREAMS; ++i) {
        if ((e = cudaEventRecord(hp.join[i], hp.s[i])) != cudaSuccess) return cuda_fail(e, "event record");
        if ((e = cudaStreamWaitEvent(s, hp.join[i], 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
    }
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return cuda_fail(e, "stream sync");
    if (trace) {
        const auto t_host2 = std::chrono::steady_clock::now();
        --trace_left;
        fprintf(stderr, "[pcgrl host trace] %lld envs, %d chunks, enqueue %.1f us, enqueue + sync %.1f us; per chunk (us from the fork):"
                        " upload done | kernels done | download done\n", (long long)n, chunks,
                std::chrono::duration<double, std::micro>(t_host1 - t_host0).count(),
                std::chrono::duration<double, std::micro>(t_host2 - t_host0).count());
        for (int c = 0; c < chunks; ++c) {
            float t[3] = {0, 0, 0};
            for (int k = 0; k < 3; ++k) cudaEventElapsedTime(&t[k], trace[3 * WL_CHUNKS], trace[3 * c + k]);
            fprintf(stderr, "[pcgrl host trace]   chunk %d (stream %d): %8.1f | %8.1f | %8.1f\n", c, c % pipe_compute(),
                    t[0] * 1e3f, t[1] * 1e3f, t[2] * 1e3f);
        }
    }
    return 0;
}

int32_t pcgrl_step_host(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions_host, void* actions_dev,
                        int64_t action_bytes, float* reward_host, uint8_t* done_host, int32_t* stats_host,
                        void* stream) {
    return step_host_impl(cfg, st, actions_host, actions_dev, action_bytes, reward_host, done_host, stats_host, nullptr,
                          stream);
}

int32_t pcgrl_step_host_packed(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions_host,
                               void* actions_dev, int64_t action_bytes, void* records_host, void* stream) {
    if (!records_host) return fail(PCGRL_E_ARG, "records_host is NULL");
    return step_host_impl(cfg, st, actions_host, actions_dev, action_bytes, nullptr, nullptr, nullptr,
                          (uint8_t*)records_host, stream);
}

}  // extern "C"
