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
#include "env_rows.cuh"
#include "level_distance.cuh"

namespace pcgrl {
cudaError_t launch_bitboard(const KParams& p, int problem, cudaStream_t s, bool& supported);
cudaError_t launch_bigboard(const KParams& p, int problem, cudaStream_t s, bool& supported);
cudaError_t launch_bitboard_split(const KParams& p, int problem, cudaStream_t s, StepPath path, bool& supported,
                                  int& n_launches, const int32_t* env_idx = nullptr, int64_t n_src = 0);
cudaError_t launch_bitboard_lanegroup(const KParams& p, int problem, cudaStream_t s, bool& supported);
int bitboard_cache_stride(int problem, int ndim, int d0, int d1, int rep, int action_kind);
cudaError_t launch_maze3d(const KParams& p, cudaStream_t s, bool& supported);
cudaError_t launch_maze3d_holey(const KParams& p, int problem, cudaStream_t s, bool& supported);
cudaError_t launch_sokoban(const KParams& p, cudaStream_t s, bool& supported);
cudaError_t launch_smb(const KParams& p, cudaStream_t s, bool& supported, int& n_launches);
int64_t sokoban_scratch_bytes();
int64_t smb_scratch_bytes(int64_t n_envs);
int64_t maze3d_scratch_bytes();
cudaError_t launch_observe(const pcgrl_config& cfg, const pcgrl_state& st, const pcgrl_obs_args& o, cudaStream_t s,
                           const int32_t* env_idx, int64_t n_idx);
const char* obs_args_error(const pcgrl_config& cfg, const pcgrl_state& st, const pcgrl_obs_args& a);
cudaError_t launch_update(const KParams& p, cudaStream_t s);
cudaError_t launch_lookahead_inc(const KParams& p, const LaOut& o, cudaStream_t s);
cudaError_t launch_lookahead_gather(const pcgrl_state& shard, const pcgrl_state& sub, const int32_t* env_idx,
                                    int row_stride, int K, int hole_ints, bool targets_per_env, int rec_stride,
                                    int status_bit, cudaStream_t s);
cudaError_t launch_step_envs_scatter(const pcgrl_state& shard, const pcgrl_state& sub, const int32_t* env_idx,
                                     int row_stride, int K, int rec_stride, cudaStream_t s);
cudaError_t launch_lookahead_apply(const KParams& p, const int32_t* env_idx, int64_t n_src, cudaStream_t s);

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
// The step path of a bit-board shard (StepPath).
// PCGRL_STEP_PATH = fused | split | inc | incfused | lg (default by shard size, below): which of the equivalent step paths
// pcgrl_step takes when the caller supplied the buffers for all of them (A/B runs and the path-equivalence tests).
// Measured on B200, binary 16x16, ms per step of a shard of 64 Ki / 256 Ki / 512 Ki / 1 Mi envs:
//   fused 0.066 / 0.131 / 0.220 / 0.385   inc (3 launches) 0.063 / 0.114 / 0.175 / 0.304   incfused 0.058 / 0.122 / 0.203 / 0.367
// so a plain pcgrl_step takes the one-launch incremental kernel for small shards and the three-launch one above.
// The lane-group kernel (step_lanegroup.cu, "lg"; kernel times, profiles/r02_lanegroup_by_size.txt): 1 Ki / 4 Ki / 16 Ki
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
// Chunks of the host pipeline (host_chunk) run on different streams.  With the search kernel of the three-launch incremental
// path limited to 3 CTAs per SM (INC_CTAS_PER_SM_HOST, step_split.cu) the memory-bound update / output kernels of the
// neighbouring chunks run NEXT TO it: e2e 2.60e9 env-steps/s at 4 chunks, against 2.24e9 with the fused kernel and
// 2.11e9 when the search holds every SM for itself (8 CTAs per SM).  The one-launch incremental kernel lost too: e2e
// 2.74e9 against at most 2.38e9 (profiles/r02_e2e_hostpath.txt).  Shards without a search cache keep the fused kernel.
// PCGRL_STEP_PATH does not apply to host-pipeline chunks.
static StepPath step_path(int64_t n_envs, int problem, bool has_cache, bool host_chunk) {
    if (host_chunk) return has_cache ? INC : FUSED;
    const StepPath dflt = problem == PCGRL_PROB_ZELDA ? FUSED
                        : !has_cache ? (n_envs < (128 << 10) ? FUSED : SPLIT)
                        : n_envs < (24 << 10) ? LANEGROUP : n_envs < (224 << 10) ? INC_FUSED : INC;
    const char* e = getenv("PCGRL_STEP_PATH");
    if (!e) return dflt;
    return !strcmp(e, "fused") ? FUSED : !strcmp(e, "split") ? SPLIT : !strcmp(e, "inc") ? INC
         : !strcmp(e, "incfused") ? INC_FUSED : !strcmp(e, "lg") ? LANEGROUP : dflt;
}
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

static int run(const KParams& p, int cfg_problem, void* stream) {
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
        // the fallback chain of StepPath: lane groups, the split path, the fused kernel, warp-per-grid boards
        StepPath path = step_path(p.n_envs, problem, p.cache != nullptr, p.host_chunk != 0);
        if (p.mode == MODE_STEP && path == LANEGROUP) {
            if (p.cache) {
                e = launch_bitboard_lanegroup(p, problem, (cudaStream_t)stream, supported);
                if (supported) {
                    if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
                    g_launches.fetch_add(1, std::memory_order_relaxed);
                    return 0;
                }
            }
            path = INC_FUSED;
        }
        if (p.mode == MODE_STEP && p.worklist && path != FUSED) {
            int n_launches = 0;
            e = launch_bitboard_split(p, problem, (cudaStream_t)stream, path, supported, n_launches);
            if (supported) {
                if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
                g_launches.fetch_add(n_launches, std::memory_order_relaxed);
                return 0;
            }
        }
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
// Streams the chunks' kernels rotate over: 3 beat 4 and 6 (e2e at 4 / 6 chunks: 2.73 / 2.76e9 with 3 streams, 2.48 /
// 2.72e9 with 4, 2.37 / 2.43e9 with 6, profiles/r02_e2e_streams.txt)
constexpr int PIPE_COMPUTE = 3;
constexpr int PIPE_STREAMS = PIPE_COMPUTE + 2;  // + one upload stream and one download stream (the last two)
struct HostGraphKey {            // everything the queued operations depend on (compared bytewise)
    pcgrl_config cfg;
    pcgrl_state st;
    void* actions_dev;
    int64_t action_bytes;
    int64_t has_host_actions;
    void *reward_host, *done_host, *stats_host, *records_host;
    int32_t chunks;
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

static int host_chunks(const pcgrl_config* cfg, int64_t n) {
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
// Layout of the work buffer of the lookahead (n candidates), of pcgrl_step_envs (n envs, `step`) and of
// pcgrl_lookahead_obs (n candidates, `obs`).  The first 256 bytes hold the work-list header of the incremental lookahead
// (only that path touches them).  Behind them, either the incremental lookahead's work-list body or the generic path's
// solver scratch (at a fixed offset: it keeps generation counters from call to call, so one zero-filled buffer serves
// every call) and the sub-shard.  The step's sub-shard also holds the outputs it writes back: stats, reward, done,
// changed and the packed records.  The observation needs the sub-shard beside the incremental path's body, so there the
// body goes behind the sub-shard.
struct LaLayout {
    int64_t inc_body, scratch, grids, mask, pos, n_step, iteration, changes, targets, holes;
    int64_t stats, reward, done, changed, records, total;
};
static int64_t la_align(int64_t x) { return (x + 255) / 256 * 256; }
static LaLayout la_layout(const pcgrl_config* c, int64_t n, bool step = false, bool obs = false) {
    LaLayout l;
    const int64_t K = c->n_stats;
    const int64_t inc_bytes = cache_stride(c) > 0 ? (2 + K + 1) * 4 * n : 0;
    l.inc_body = 256;
    const int64_t inc_end = inc_bytes ? l.inc_body + la_align(inc_bytes) : 0;
    l.scratch = 256;
    int64_t off = l.scratch + la_align(pcgrl_scratch_bytes(c, n));
    auto take = [&](int64_t bytes) {
        const int64_t at = off;
        off += la_align(bytes);
        return at;
    };
    l.grids = take(n * c->row_stride);
    l.mask = take(n * c->row_stride);
    l.pos = take(n * 12);
    l.n_step = take(n * 4);
    l.iteration = take(n * 4);
    l.changes = take(n * 4);
    l.targets = take(c->targets_per_env ? n * K * 16 : 0);
    l.holes = take(is_holey(c) ? n * hole_ints(c) * 4 : 0);
    l.stats = take(step ? n * K * 4 : 0);
    l.reward = take(step ? n * 4 : 0);
    l.done = take(step ? n : 0);
    l.changed = take(step ? n : 0);
    l.records = take(step ? n * record_stride(c) : 0);
    if (obs) l.inc_body = take(inc_bytes);
    l.total = step || obs ? off : std::max(off, inc_end);
    return l;
}

// The packed env row of pcgrl_save_envs / pcgrl_load_envs (format in include/pcgrl_b200.h), decided here and nowhere
// else: the offsets for the caller, and (rc != NULL) the pieces the copy kernels move.  The shard's arguments have been
// checked.
static int32_t env_row_layout(const pcgrl_config* c, const pcgrl_state* st, int32_t n_pos, pcgrl_row_layout* l,
                              RowCopy* rc) {
    const int64_t K = c->n_stats, rs = c->row_stride;
    std::memset(l, 0, sizeof(*l));
    l->n_pos = n_pos;
    if (rc) std::memset(rc, 0, sizeof(*rc));
    int64_t off = 16;                  // the header
    uint32_t h = 2166136261u;          // FNV-1a over the fields that give the row's bytes their meaning
    auto mix = [&](int64_t v) {
        for (int b = 0; b < 8; ++b) h = (h ^ (uint32_t)((uint64_t)v >> (8 * b) & 0xff)) * 16777619u;
    };
    // a section of `bytes` bytes (0: absent, offset -1) at the next 16-byte boundary
    auto section = [&](int64_t bytes) -> int32_t {
        mix(bytes);
        if (!bytes) return -1;
        const int64_t at = off;
        off += (bytes + 15) / 16 * 16;
        return (int32_t)at;
    };
    auto piece = [&](int32_t at, const void* base, int64_t item, int64_t count, int64_t item_stride) {
        if (!rc || at < 0) return;
        RowPiece& q = rc->piece[rc->n_pieces++];
        q.base = const_cast<void*>(base);
        q.off = at;
        q.item = (int32_t)item;
        q.count = (int32_t)count;
        q.item_stride = item_stride;
        const uint64_t m = (uint64_t)at | (uint64_t)item | (uintptr_t)base | (count > 1 ? (uint64_t)item_stride : 0) | 16;
        q.unit = (int32_t)(m & (~m + 1));   // the lowest set bit
    };
    for (const int64_t v : {c->problem, c->representation, c->action_kind, c->ndim, c->n_tiles, c->n_stats, c->row_stride})
        mix(v);
    for (int i = 0; i < 3; ++i) mix(i < c->ndim ? c->dims[i] : 1);
    const int64_t cs = st->worklist && st->cache ? cache_stride(c) : 0;   // the condition fill() uses
    const int64_t rec = c->record_stat_bytes && st->records ? record_stride(c) : 0;
    const int64_t hi = is_holey(c) ? hole_ints(c) : 0;
    piece(l->grid = section(rs), st->grids, rs, 1, 0);
    piece(l->static_mask = section(st->static_mask ? rs : 0), st->static_mask, rs, 1, 0);
    piece(l->cache = section(cs), st->cache, cs, 1, 0);
    piece(l->records = section(rec), st->records, rec, 1, 0);
    piece(l->targets = section(c->targets_per_env ? 16 * K : 0), st->targets, 16 * K, 1, 0);
    piece(l->stats = section(4 * K), st->stats, 4 * K, 1, 0);
    piece(l->holes = section(4 * hi), st->holes, 4 * hi, 1, 0);
    piece(l->pos = section(12 * (int64_t)n_pos), st->pos, 12, n_pos, 12 * st->n_envs);   // agent a's array: pos + a * N * 3
    l->n_step = section(12);
    l->iteration = l->n_step + 4;
    l->changes = l->n_step + 8;
    piece(l->n_step, st->n_step, 4, 1, 0);
    piece(l->iteration, st->iteration, 4, 1, 0);
    piece(l->changes, st->changes, 4, 1, 0);
    l->reward = section(st->changed ? 6 : 5);
    l->done = l->reward + 4;
    l->changed = st->changed ? l->reward + 5 : -1;
    piece(l->reward, st->reward, 4, 1, 0);
    piece(l->done, st->done, 1, 1, 0);
    piece(l->changed, st->changed, 1, 1, 0);
    if (off > INT32_MAX) return fail(PCGRL_E_ARG, "row too large (n_pos)");
    l->row_bytes = (int32_t)off;
    l->signature = h ? h : 1;          // an all-zero header is never valid
    if (rc) {
        rc->row_bytes = l->row_bytes;
        rc->signature = l->signature;
        rc->n_envs = st->n_envs;
        rc->status = st->status;
    }
    return 0;
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
// parent's buffer, host_chunk = true); a plain pcgrl_step is chunk 0 at offset 0 of its own buffer.
static int32_t step_launch(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions, void* stream,
                           int32_t* wl_base, int wl_chunk, int64_t wl_off, bool host_chunk = false) {
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
    p.host_chunk = host_chunk;
    return run(p, cfg->problem, stream);
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

// Shared body of pcgrl_observe / pcgrl_observe_envs (env_idx NULL: every env of the shard).
static int32_t observe_impl(const pcgrl_config* cfg, const pcgrl_state* st, const pcgrl_obs_args* obs,
                            const int32_t* env_idx, int64_t n_idx, void* stream) {
    int r = check(cfg);
    if (r) return r;
    if (!st || !st->grids || !st->pos || !obs || !obs->out) return fail(PCGRL_E_ARG, "bad observe arguments");
    if (obs->n_ctrl < 0 || obs->n_ctrl > PCGRL_MAX_STATS) return fail(PCGRL_E_ARG, "n_ctrl out of range");
    if (obs->n_ctrl > 0 && (!st->stats || !st->targets)) return fail(PCGRL_E_ARG, "control channels need stats/targets");
    cudaError_t e = launch_observe(*cfg, *st, *obs, (cudaStream_t)stream, env_idx, n_idx);
    if (e != cudaSuccess) return cuda_fail(e, "observe launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

int32_t pcgrl_observe(const pcgrl_config* cfg, const pcgrl_state* st, const pcgrl_obs_args* obs, void* stream) {
    return observe_impl(cfg, st, obs, nullptr, 0, stream);
}

int32_t pcgrl_observe_envs(const pcgrl_config* cfg, const pcgrl_state* st, const pcgrl_obs_args* obs,
                           const int32_t* env_idx, int64_t n_idx, void* stream) {
    if (n_idx < 0) return fail(PCGRL_E_ARG, "n_idx < 0");
    if (n_idx > 0 && !env_idx) return fail(PCGRL_E_ARG, "env_idx is NULL");
    int r = check(cfg);
    if (r) return r;
    if (!st || !obs) return fail(PCGRL_E_ARG, "bad observe arguments");
    if (n_idx == 0) return 0;   // nothing to write, nothing launched
    return observe_impl(cfg, st, obs, env_idx, n_idx, stream);
}

// The generic path's sub-shard of n envs inside `work` (layout l): grids, frozen mask, pos, counters, per-env targets,
// holes and solver scratch.  The caller points stats / reward / done / changed / records.
static pcgrl_state sub_shard(const pcgrl_config* cfg, const pcgrl_state* st, int64_t n, uint8_t* w, const LaLayout& l) {
    pcgrl_state sub;
    std::memset(&sub, 0, sizeof(sub));
    sub.n_envs = n;
    sub.env_offset = st->env_offset;
    sub.grids = (int8_t*)(w + l.grids);
    sub.static_mask = st->static_mask ? w + l.mask : nullptr;
    sub.pos = (int32_t*)(w + l.pos);
    sub.n_step = (int32_t*)(w + l.n_step);
    sub.iteration = (int32_t*)(w + l.iteration);
    sub.changes = (int32_t*)(w + l.changes);
    sub.targets = cfg->targets_per_env ? (const double*)(w + l.targets) : st->targets;
    sub.holes = st->holes && is_holey(cfg) ? (int32_t*)(w + l.holes) : nullptr;
    sub.status = st->status;
    sub.scratch = pcgrl_scratch_bytes(cfg, n) > 0 ? w + l.scratch : nullptr;
    return sub;
}

int64_t pcgrl_lookahead_work_bytes(const pcgrl_config* cfg, int64_t n) {
    if (check(cfg) || n < 0) return -1;
    return la_layout(cfg, n).total;
}

int64_t pcgrl_lookahead_obs_work_bytes(const pcgrl_config* cfg, int64_t n) {
    if (check(cfg) || n < 0) return -1;
    return la_layout(cfg, n, false, true).total;
}

// Shared body of pcgrl_lookahead (obs NULL) and pcgrl_lookahead_obs: every check before any CUDA call.
static int32_t lookahead_impl(const pcgrl_config* cfg, const pcgrl_state* st, const pcgrl_obs_args* obs,
                              const void* actions, const int32_t* env_idx, int64_t n, float* reward, uint8_t* done,
                              uint8_t* changed, int32_t* stats, void* work, void* stream) {
    int r = check(cfg);
    if (r) return r;
    if ((r = check_state(st))) return r;
    if (n < 0 || n > INT32_MAX) return fail(PCGRL_E_ARG, "n must be in [0, 2^31)");
    if (!env_idx && n > st->n_envs) return fail(PCGRL_E_ARG, "without env_idx candidate j is env j: n > n_envs");
    if (n > 0 && (!actions || !reward || !done || !changed || !stats || !work))
        return fail(PCGRL_E_ARG, "actions, reward, done, changed, stats and work must not be NULL");
    if (is_holey(cfg) && !st->holes) return fail(PCGRL_E_ARG, "a holey problem needs pcgrl_state.holes");
    if (obs) {
        if (n > 0 && !obs->out) return fail(PCGRL_E_ARG, "obs->out is NULL");
        if (obs->n_ctrl < 0 || obs->n_ctrl > PCGRL_MAX_STATS) return fail(PCGRL_E_ARG, "n_ctrl out of range");
        if ((obs->out_kind < 0 || obs->out_kind > 3) && obs->out_kind != 5 && obs->out_kind != 6)
            return fail(PCGRL_E_ARG, "out_kind out of range");
        if (const char* m = obs_args_error(*cfg, *st, *obs)) return fail(PCGRL_E_ARG, m);
    }
    if (n == 0) return 0;   // nothing to write, nothing launched
    KParams p;
    fill(p, cfg, st);
    uint8_t* w = (uint8_t*)work;
    const cudaStream_t s = (cudaStream_t)stream;
    const LaLayout l = la_layout(cfg, n, false, obs != nullptr);
    // the candidates' rows as a sub-shard of n envs; the lookahead's outputs are its stats / reward / done / changed
    pcgrl_state sub = sub_shard(cfg, st, n, w, l);
    sub.stats = stats;
    sub.reward = reward;
    sub.done = done;
    sub.changed = changed;
    auto gather = [&]() {
        const cudaError_t e = launch_lookahead_gather(*st, sub, env_idx, cfg->row_stride, cfg->n_stats, hole_ints(cfg),
                                                      cfg->targets_per_env != 0, 0, 128, s);
        if (e != cudaSuccess) return cuda_fail(e, "lookahead gather launch");
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return 0;
    };
    cudaError_t e;
    if (p.cache) {   // the shard keeps a search cache: incremental searches from it
        // the observation's copy of e's rows first: the gather writes e's old stats, the incremental path the new ones
        if (obs && (r = gather())) return r;
        LaOut o{env_idx, st->n_envs, reward, done, changed, stats};
        p.mode = MODE_STEP;
        p.actions = actions;
        p.n_envs = n;
        p.records = nullptr;
        p.wl_hdr = (int32_t*)w;
        p.worklist = (int32_t*)(w + l.inc_body);
        if ((e = launch_lookahead_inc(p, o, s)) != cudaSuccess) return cuda_fail(e, "lookahead launch");
        g_launches.fetch_add(3, std::memory_order_relaxed);
        if (!obs) return 0;
        // the candidate's edit and position advance, on the copy
        KParams q;
        fill(q, cfg, &sub);
        q.mode = MODE_STEP;
        q.actions = actions;
        if ((e = launch_lookahead_apply(q, env_idx, st->n_envs, s)) != cudaSuccess)
            return cuda_fail(e, "lookahead apply launch");
        g_launches.fetch_add(1, std::memory_order_relaxed);
    } else {   // every other config: the ordinary step on the sub-shard
        if ((r = gather())) return r;
        if ((r = step_launch(cfg, &sub, actions, stream, nullptr, 0, 0))) return r;
        if (!obs) return 0;
    }
    // the after-states are rows 0..n-1 of the sub-shard: the unchanged observation writer on it
    if ((e = launch_observe(*cfg, sub, *obs, s, nullptr, 0)) != cudaSuccess) return cuda_fail(e, "observe launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

int32_t pcgrl_lookahead(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions, const int32_t* env_idx,
                        int64_t n, float* reward, uint8_t* done, uint8_t* changed, int32_t* stats, void* work,
                        void* stream) {
    return lookahead_impl(cfg, st, nullptr, actions, env_idx, n, reward, done, changed, stats, work, stream);
}

int32_t pcgrl_lookahead_obs(const pcgrl_config* cfg, const pcgrl_state* st, const pcgrl_obs_args* obs,
                            const void* actions, const int32_t* env_idx, int64_t n, float* reward, uint8_t* done,
                            uint8_t* changed, int32_t* stats, void* work, void* stream) {
    if (!obs) return fail(PCGRL_E_ARG, "obs is NULL");
    return lookahead_impl(cfg, st, obs, actions, env_idx, n, reward, done, changed, stats, work, stream);
}

int64_t pcgrl_step_envs_work_bytes(const pcgrl_config* cfg, int64_t n) {
    if (check(cfg) || n < 0) return -1;
    return la_layout(cfg, n, true).total;
}

int32_t pcgrl_step_envs(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions, const int32_t* env_idx,
                        int64_t n, void* work, void* stream) {
    int r = check(cfg);
    if (r) return r;
    if ((r = check_state(st))) return r;
    if (n < 0 || n > INT32_MAX) return fail(PCGRL_E_ARG, "n must be in [0, 2^31)");
    if (n > st->n_envs) return fail(PCGRL_E_ARG, "n distinct env indices: n > n_envs");
    if (n > 0 && (!actions || !env_idx || !work)) return fail(PCGRL_E_ARG, "actions, env_idx and work must not be NULL");
    if (is_holey(cfg) && !st->holes) return fail(PCGRL_E_ARG, "a holey problem needs pcgrl_state.holes");
    if (n == 0) return 0;   // nothing to write, nothing launched
    KParams p;
    fill(p, cfg, st);
    p.mode = MODE_STEP;
    p.actions = actions;
    p.n_envs = n;
    const cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e;
    if (p.worklist) {   // the split path's three launches through the shard's own work list (chunk 0's header)
        bool supported = false;
        int n_launches = 0;
        e = launch_bitboard_split(p, kernel_problem(cfg->problem), s, INC, supported, n_launches, env_idx, st->n_envs);
        if (supported) {
            if (e != cudaSuccess) return cuda_fail(e, "step_envs launch");
            g_launches.fetch_add(n_launches, std::memory_order_relaxed);
            return 0;
        }
    }
    // every other config: the listed rows as a sub-shard of n envs, the ordinary step on it, and the rows back
    uint8_t* w = (uint8_t*)work;
    const LaLayout l = la_layout(cfg, n, true);
    pcgrl_state sub = sub_shard(cfg, st, n, w, l);
    sub.stats = (int32_t*)(w + l.stats);
    sub.reward = (float*)(w + l.reward);
    sub.done = w + l.done;
    sub.changed = w + l.changed;
    sub.records = p.records ? w + l.records : nullptr;
    const int rs = p.records ? record_stride(cfg) : 0;
    if ((e = launch_lookahead_gather(*st, sub, env_idx, cfg->row_stride, cfg->n_stats, hole_ints(cfg),
                                     cfg->targets_per_env != 0, rs, 256, s)) != cudaSuccess)
        return cuda_fail(e, "step_envs gather launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if ((r = step_launch(cfg, &sub, actions, stream, nullptr, 0, 0))) return r;
    if ((e = launch_step_envs_scatter(*st, sub, env_idx, cfg->row_stride, cfg->n_stats, rs, s)) != cudaSuccess)
        return cuda_fail(e, "step_envs scatter launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

static int32_t check_rows_shard(const pcgrl_config* cfg, const pcgrl_state* st, int32_t n_pos) {
    int r = check(cfg);
    if (r) return r;
    if ((r = check_state(st))) return r;
    if (n_pos < 1) return fail(PCGRL_E_ARG, "n_pos must be >= 1");
    if (is_holey(cfg) && !st->holes) return fail(PCGRL_E_ARG, "a holey problem needs pcgrl_state.holes");
    return 0;
}

int32_t pcgrl_env_row_layout(const pcgrl_config* cfg, const pcgrl_state* st, int32_t n_pos, pcgrl_row_layout* out) {
    int r = check_rows_shard(cfg, st, n_pos);
    if (r) return r;
    if (!out) return fail(PCGRL_E_ARG, "out is NULL");
    return env_row_layout(cfg, st, n_pos, out, nullptr);
}

// Shared body of pcgrl_save_envs / pcgrl_load_envs: every check before any CUDA call, then one launch.
static int32_t env_rows_impl(const pcgrl_config* cfg, const pcgrl_state* st, int32_t n_pos, const void* rows,
                             const int32_t* env_idx, int64_t n, void* stream, bool save) {
    int r = check_rows_shard(cfg, st, n_pos);
    if (r) return r;
    if (n < 0 || n > INT32_MAX) return fail(PCGRL_E_ARG, "n must be in [0, 2^31)");
    if (!env_idx && n > st->n_envs) return fail(PCGRL_E_ARG, "without env_idx row j is env j: n > n_envs");
    if (!save && n > st->n_envs) return fail(PCGRL_E_ARG, "load: n distinct env indices: n > n_envs");
    if (n > 0 && !rows) return fail(PCGRL_E_ARG, "rows is NULL");
    if ((uintptr_t)rows % 16) return fail(PCGRL_E_ARG, "rows must be 16-byte aligned");
    pcgrl_row_layout l;
    RowCopy rc;
    if ((r = env_row_layout(cfg, st, n_pos, &l, &rc))) return r;
    if (n * (l.row_bytes / 16) / 256 >= INT32_MAX) return fail(PCGRL_E_ARG, "too many rows for one launch");
    if (n == 0) return 0;   // nothing to write, nothing launched
    rc.rows = (uint8_t*)const_cast<void*>(rows);
    rc.env_idx = env_idx;
    rc.n_rows = n;
    const cudaError_t e = save ? launch_save_envs(rc, (cudaStream_t)stream) : launch_load_envs(rc, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, save ? "save_envs launch" : "load_envs launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

int32_t pcgrl_save_envs(const pcgrl_config* cfg, const pcgrl_state* st, int32_t n_pos, const int32_t* env_idx,
                        int64_t n, void* rows, void* stream) {
    return env_rows_impl(cfg, st, n_pos, rows, env_idx, n, stream, true);
}

int32_t pcgrl_load_envs(const pcgrl_config* cfg, const pcgrl_state* st, int32_t n_pos, const void* rows,
                        const int32_t* env_idx, int64_t n, void* stream) {
    return env_rows_impl(cfg, st, n_pos, rows, env_idx, n, stream, false);
}

// ---- level distances: every check before any CUDA call ------------------------------------------------------------
static int32_t check_levels(const LdGeom& g, const void* p, int64_t n, int64_t stride, const char* what) {
    if (n < 0 || n > INT32_MAX) return fail(PCGRL_E_ARG, std::string(what) + ": count must be in [0, 2^31)");
    if (stride < g.cells) return fail(PCGRL_E_ARG, std::string(what) + ": stride must be >= cells");
    if (n > 0 && !p) return fail(PCGRL_E_ARG, std::string(what) + " is NULL");
    if (n * g.W / 8 >= INT32_MAX) return fail(PCGRL_E_ARG, std::string(what) + ": too many levels for one launch");
    return 0;
}

static int32_t check_level_call(const pcgrl_config* cfg, LdGeom& g, const void* work) {
    const int r = check(cfg);
    if (r) return r;
    g = ld_geom(cells_of(cfg), cfg->n_tiles);
    if (!ld_fits(g)) return fail(PCGRL_E_UNSUPPORTED, "level too large for the distance tile's shared memory");
    if (!work) return fail(PCGRL_E_ARG, "work is NULL");
    if ((uintptr_t)work % 16) return fail(PCGRL_E_ARG, "work must be 16-byte aligned");
    return 0;
}

int64_t pcgrl_level_work_bytes(const pcgrl_config* cfg, int64_t n_query, int64_t n_archive, int32_t k) {
    if (check(cfg) || n_query < 0 || n_archive < 0 || k < 0 || k > 64) return -1;
    return ld_work_bytes(ld_geom(cells_of(cfg), cfg->n_tiles), n_query, n_archive, k);
}

int32_t pcgrl_level_distances(const pcgrl_config* cfg, const void* a, int64_t n_a, int64_t a_stride, const void* b,
                              int64_t n_b, int64_t b_stride, int32_t* out, void* work, void* stream) {
    LdGeom g;
    int r;
    if ((r = check_level_call(cfg, g, work)) || (r = check_levels(g, a, n_a, a_stride, "a")) ||
        (r = check_levels(g, b, n_b, b_stride, "b")))
        return r;
    if (n_a > 0 && n_b > 0 && !out) return fail(PCGRL_E_ARG, "out is NULL");
    if (n_a == 0 || n_b == 0) return 0;
    int launches = 0;
    const cudaError_t e = launch_level_distances(g, {(const uint8_t*)a, n_a, a_stride}, {(const uint8_t*)b, n_b, b_stride},
                                                 out, work, (cudaStream_t)stream, launches);
    g_launches.fetch_add(launches, std::memory_order_relaxed);
    return e == cudaSuccess ? 0 : cuda_fail(e, "level_distances launch");
}

int32_t pcgrl_level_knn(const pcgrl_config* cfg, const void* q, int64_t n_q, int64_t q_stride, const void* b,
                        int64_t n_b, int64_t b_stride, int32_t k, int64_t self_offset, int32_t* dist, int32_t* idx,
                        void* work, void* stream) {
    LdGeom g;
    int r;
    if ((r = check_level_call(cfg, g, work)) || (r = check_levels(g, q, n_q, q_stride, "queries")) ||
        (r = check_levels(g, b, n_b, b_stride, "archive")))
        return r;
    if (k < 1 || k > 64) return fail(PCGRL_E_ARG, "k must be in [1, 64]");
    if (self_offset < -1) return fail(PCGRL_E_ARG, "self_offset must be >= -1 (-1: no self-exclusion)");
    if (n_q > 0 && (!dist || !idx)) return fail(PCGRL_E_ARG, "dist / idx is NULL");
    if (n_q == 0) return 0;
    int launches = 0;
    const cudaError_t e = launch_level_knn(g, {(const uint8_t*)q, n_q, q_stride}, {(const uint8_t*)b, n_b, b_stride}, k,
                                           self_offset, dist, idx, work, (cudaStream_t)stream, launches);
    g_launches.fetch_add(launches, std::memory_order_relaxed);
    return e == cudaSuccess ? 0 : cuda_fail(e, "level_knn launch");
}

int32_t pcgrl_level_group_diversity(const pcgrl_config* cfg, const void* a, int64_t n, int64_t stride,
                                    int64_t group_size, int64_t* sums, void* work, void* stream) {
    LdGeom g;
    int r;
    if ((r = check_level_call(cfg, g, work)) || (r = check_levels(g, a, n, stride, "levels"))) return r;
    if (group_size < 2) return fail(PCGRL_E_ARG, "group_size must be >= 2");
    if (n % group_size) return fail(PCGRL_E_ARG, "group_size must divide the level count");
    if (n > 0 && !sums) return fail(PCGRL_E_ARG, "sums is NULL");
    if (n == 0) return 0;
    int launches = 0;
    const cudaError_t e = launch_level_groups(g, {(const uint8_t*)a, n, stride}, group_size, sums, work,
                                              (cudaStream_t)stream, launches);
    g_launches.fetch_add(launches, std::memory_order_relaxed);
    return e == cudaSuccess ? 0 : cuda_fail(e, "level_group_diversity launch");
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
    const int chunks = (n > 0 && (!actions_host || action_bytes % n == 0)) ? host_chunks(cfg, n) : 1;
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
    // kernels starting 60 us after the first chunk's had ended.)
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
        cudaStream_t up = hp.s[PIPE_COMPUTE], down = hp.s[PIPE_COMPUTE + 1];
        // every upload first: 1 B per env, on its own stream, long before the chunk's turn comes
        for (int c = 0; c < n_ck && actions_host; ++c) {
            if ((e = cudaMemcpyAsync(ck[c].a_dev, (const char*)actions_host + ck[c].off * a_env, (size_t)(ck[c].m * a_env),
                                     cudaMemcpyHostToDevice, up)) != cudaSuccess)
                return cuda_fail(e, "H2D actions");
            if ((e = cudaEventRecord(hp.up_ev[c], up)) != cudaSuccess) return cuda_fail(e, "event record");
            if (trace) cudaEventRecord(trace[3 * c + 0], up);
        }
        for (int c = 0; c < n_ck; ++c) {
            const int64_t off = ck[c].off, m = ck[c].m;
            const pcgrl_state& sub = ck[c].sub;
            cudaStream_t cs = hp.s[c % PIPE_COMPUTE];
            if (actions_host) {
                if ((e = cudaStreamWaitEvent(cs, hp.up_ev[c], 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
            } else if (trace) {
                cudaEventRecord(trace[3 * c + 0], cs);
            }
            // every chunk gets its own header and its own body range of the shard's work list
            int rr = step_launch(cfg, &sub, ck[c].a_dev, cs, st->worklist, c, off, true);
            if (rr) return rr;
            if (trace) cudaEventRecord(trace[3 * c + 1], cs);
            if ((e = cudaEventRecord(hp.k_ev[c], cs)) != cudaSuccess) return cuda_fail(e, "event record");
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
    };

    // ---- CUDA graph of the whole pipeline -------------------------------------------------------------------------
    // A step of the host pipeline is ~25 queue operations (copies, launches, events over five streams) whose CPU cost sits
    // on the critical path of every step: the first kernel cannot start before its upload is queued, and the call
    // cannot return before the last event is.  The operations only depend on the pointers, so they are captured ONCE
    // (stream capture on helper stream 0, the others forked / joined by events inside the capture) and replayed
    // with one cudaGraphLaunch; only the source addresses of the uploads change from step to step
    // (cudaGraphExecMemcpyNodeSetParams1D).  Tracing, and a driver that cannot capture the pipeline, queue the
    // operations directly (below).
    if (!hp.graph_broken && !trace) {
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
            fprintf(stderr, "[pcgrl host trace]   chunk %d (stream %d): %8.1f | %8.1f | %8.1f\n", c, c % PIPE_COMPUTE,
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
