/*
 * pcgrl_b200.h -- C ABI of libpcgrl_sm100.so: the batched, B200-native PCGRL environment step.
 *
 * This is the drop-in boundary for ONE hot path of smearle/control-pcgrl: env.step() for thousands of
 * level grids at once (representation update -> problem get_stats -> ControlWrapper reward).
 * The reference has no native layer (it is 100 % Python), so there is no existing FFI to mirror;
 * each entry point below names the reference Python interface it replaces (paths relative to
 * /root/reference/control_pcgrl/).  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *   - plain C types only; every pointer in the *_args structs is a DEVICE pointer owned by the caller
 *     (PyTorch tensors in the Python host), except where a field says "host".
 *   - launches are asynchronous on the `stream` argument (a cudaStream_t passed as void*).
 *   - the library keeps no global state except a thread-local last-error string; it allocates no
 *     device memory: callers size scratch with pcgrl_scratch_bytes() and pass it in.
 *   - return value: 0 = ok, negative = error (PCGRL_E_*); pcgrl_last_error() gives the message.
 *     Nothing throws across the ABI.  There is no CPU fallback: without a CUDA device every launch
 *     entry point returns PCGRL_E_CUDA.
 */
#ifndef PCGRL_B200_H
#define PCGRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCGRL_ABI_VERSION 5

/* problems: envs/probs/__init__.py:31-58 (the five BASELINE.json names) */
enum { PCGRL_PROB_BINARY = 0, PCGRL_PROB_ZELDA = 1, PCGRL_PROB_SOKOBAN = 2, PCGRL_PROB_SMB = 3,
       PCGRL_PROB_MINECRAFT_3D_MAZE = 4,
       /* SURVEY 8f rank 2 -- holey problems: stats on the bordered map with an entrance and an exit dug into the
          border (envs/probs/binary/binary_holey_prob.py:59-93, envs/pcgrl_holey_env.py:44-53) */
       PCGRL_PROB_BINARY_HOLEY = 5,
       /* SURVEY 8f rank 4 -- minecraft_2D_maze (envs/probs/minecraft/minecraft_2D_maze_prob.py:87-93): regions and
          longest path over the "AIR" tile (code 0), i.e. the binary stats under other tile names */
       PCGRL_PROB_MINECRAFT_2D_MAZE = 6,
       /* SURVEY 8f rank 2, the 3D holey problems (envs/probs/minecraft/minecraft_3D_holey_maze_prob.py:71-130,
          minecraft_3D_holey_dungeon_prob.py:95-146, envs/probs/holey_prob_3D.py): stats on the bordered 3D map with a
          two-tile-high entrance and exit dug into its sides; maps up to 14^3.  The holey maze has FIVE stats: the four
          the reference returns plus the length found by this call, which the reference reports one call late */
       PCGRL_PROB_MINECRAFT_3D_HOLEY_MAZE = 7, PCGRL_PROB_MINECRAFT_3D_DUNGEON_HOLEY = 8 };
/* where reset takes the entrance / exit holes of a holey problem from (envs/probs/holey_prob.py:32-60 gen_holes) */
enum {
    PCGRL_HOLES_GIVEN = 0,   /* leave pcgrl_state.holes as the caller set them (the reference's _hole_queue) */
    PCGRL_HOLES_FIXED = 1,   /* fixed_holes: entrance (1, 0), exit (W, H + 1)  (holey_prob.py:47-49) */
    PCGRL_HOLES_RANDOM = 2   /* four distinct random border cells; entrance = the first, exit = the first of the
                                other three that _valid_holes accepts, else the previous exit (:51-58) */
};
/* representations: envs/reps/__init__.py:11-23 */
enum { PCGRL_REP_NARROW = 0, PCGRL_REP_TURTLE = 1, PCGRL_REP_WIDE = 2, PCGRL_REP_CELLULAR = 3 };
/* action encodings */
enum {
    PCGRL_ACT_INT32 = 0,       /* narrow/turtle: int32[N]  (Discrete, reps/narrow_rep.py:65, turtle_rep.py:70) */
    PCGRL_ACT_WIDE_COORDS = 1, /* wide: int32[N, ndim+1] = [*coords, tile]  (reps/wide_rep.py:23-24,35-40)   */
    PCGRL_ACT_WIDE_FLAT = 2,   /* wide: int32[N] flat ActionMap index over (act_h, act_w, C); writes _map[x, y]
                                  (wrappers.py:304-323)                                                      */
    PCGRL_ACT_CA_TILES = 3,    /* cellular: int8[N, row_stride] already-argmaxed next map                    */
    PCGRL_ACT_CA_LOGITS = 4,   /* cellular: float32[N, C, cells] logits; argmax over C, lowest index wins
                                  (reps/ca_rep.py:31-44, wrappers.py:157-165)                                */
    PCGRL_ACT_PATCH = 5        /* narrow + MultiActionRepresentation (cfg.act_window): int32[N, prod(act_window)]
                                  tile codes of the whole patch, C order of action.reshape(act_window)
                                  (envs/reps/wrappers.py:397-545; MultiDiscrete([C] * prod), :438-443)        */
};
/* how `reward` is computed from the old and new stats */
enum {
    PCGRL_REWARD_CONTROL = 0,  /* ControlWrapper: loss(new) - loss(old), loss = -sum w |trg - val|
                                  (control_wrappers.py:216-244, 318-345) -- what step() pays at this commit */
    PCGRL_REWARD_RANGE = 1     /* legacy Problem.get_reward: sum w * get_range_reward(new, old, lo, hi)
                                  (envs/helper.py:550-560; e.g. probs/binary/binary_prob.py:170-178); `targets`
                                  rows are read as the (lo, hi) of each stat and may hold +-infinity */
};
enum { PCGRL_E_ARG = -1, PCGRL_E_CUDA = -2, PCGRL_E_UNSUPPORTED = -3 };

#define PCGRL_MAX_STATS 16
#define PCGRL_MAX_TILES 16

/* Static description of one env shard.  Mirrors what PcgrlEnv.__init__/adjust_param derive
 * (envs/pcgrl_env.py:39-94, 221-247). */
typedef struct pcgrl_config {
    int32_t abi_version;      /* PCGRL_ABI_VERSION */
    int32_t problem;          /* PCGRL_PROB_* */
    int32_t representation;   /* PCGRL_REP_* */
    int32_t action_kind;      /* PCGRL_ACT_* */
    int32_t ndim;             /* 2 or 3 */
    int32_t dims[3];          /* 2D: {H, W, 1};  3D: {Z, Y, X} -- numpy axis order of _map */
    int32_t n_tiles;          /* C */
    int32_t n_stats;          /* K, order = the problem's get_stats dict order */
    int32_t row_stride;       /* bytes per env in `grids` (cells rounded up to a multiple of 16) */
    int32_t max_iterations;   /* pcgrl_env.py:241 */
    int32_t max_changes;      /* pcgrl_env.py:235-239; < 0 = unlimited */
    int32_t act_h, act_w;     /* PCGRL_ACT_WIDE_FLAT only: ActionMap's (h, w) (wrappers.py:283-287) */
    int32_t targets_per_env;  /* 1: targets is [N,K,2]; 0: targets is [1,K,2] shared by all envs */
    int32_t init_random_probs;/* reset: 1 = draw per-episode tile probabilities U(0,1)^C normalised
                                 (pcgrl_env.py:162-164), 0 = use init_probs as given */
    int32_t reward_mode;      /* PCGRL_REWARD_* */
    float   init_probs[PCGRL_MAX_TILES]; /* tile init distribution, normalised by the library */
    double  weights[PCGRL_MAX_STATS];    /* ControlWrapper.metric_weights per stat (0 = not in all_metrics),
                                            control_wrappers.py:41-45,78-84 */
    /* -- representation wrappers (envs/reps/wrappers.py wrap_rep :717-722), ABI 3 -------------------------- */
    int32_t act_window[3];    /* MultiActionRepresentation: size of the action patch per map axis
                                 (cfg.act_window, wrappers.py:413-417); {0,0,0} = off.  Needs PCGRL_ACT_PATCH */
    float   static_prob;      /* StaticTileRepresentation, random resets only: upper bound of the per-episode
                                 frozen-tile probability (wrappers.py:279-289); 0 = none */
    int32_t n_static_walls;   /* random resets only: number of frozen random wall segments (wrappers.py:291-308) */
    int32_t wall_tile;        /* tile code written along those walls (Problem._wall_tile, pcgrl_env.py:58) */
    int32_t static_eval_mode; /* 1: use static_prob itself instead of U(0,1)*static_prob (set_eval_mode, :268) */
    /* -- holey problems, ABI 4 --------------------------------------------------------------------------- */
    int32_t hole_mode;        /* PCGRL_HOLES_*; only read by resets of a holey problem */
    /* -- compact host I/O, ABI 5 ------------------------------------------------------------------------- */
    int32_t action_elem_bytes;/* PCGRL_ACT_INT32 / PCGRL_ACT_WIDE_FLAT only: bytes per action element, 0 or 4 = int32
                                 (the default), 1 = uint8, 2 = uint16 -- a Discrete(2) action is one byte over PCIe
                                 instead of four */
    int32_t record_stat_bytes;/* 0 = no packed result records; 1 = uint8, 2 = int16, 4 = int32 per stat in
                                 pcgrl_state.records (the host picks the narrowest type the problem's stat bounds
                                 fit; a value that does not fit sets status bit 4) */
} pcgrl_config;

/* Device-resident state of N envs + the per-step inputs/outputs.
 * Replaces: PcgrlEnv.step (envs/pcgrl_env.py:267-342), Representation.update (envs/reps/*.py),
 * Problem.get_stats (envs/probs/<game>/*_prob.py) and ControlWrapper.step/get_loss
 * (control_wrappers.py:216-244, 318-345). */
typedef struct pcgrl_state {
    int64_t  n_envs;
    int64_t  env_offset;   /* global index of env 0 of this shard (only seeds the reset RNG) */
    int8_t*  grids;        /* [N, row_stride] tile codes, row-major cells (C order of _map); in place */
    int32_t* pos;          /* [N, 3] agent position in numpy axis order (unused axes 0).  Multi-agent turtle
                              (envs/reps/wrappers.py:612-651, one env step per agent): the caller keeps one such
                              array per agent and passes the acting / observing agent's */
    int32_t* n_step;       /* [N] narrow scan counter (reps/narrow_rep.py:98-100) */
    int32_t* iteration;    /* [N] PcgrlEnv._iteration */
    int32_t* changes;      /* [N] PcgrlEnv._changes */
    int32_t* stats;        /* [N, K] current _rep_stats; read (old) and written (new) by step */
    const double* targets; /* [N or 1, K, 2] (lo, hi): hi = NaN -> scalar target lo, else the integer range
                              np.arange(lo, hi) (control_wrappers.py:336-343).  With PCGRL_REWARD_RANGE: the
                              (lo, hi) band of get_range_reward for each stat */
    float*   reward;       /* [N] out: loss(new stats) - loss(old stats), evaluated in fp64 */
    uint8_t* done;         /* [N] out: done == truncated (pcgrl_env.py:307-310) */
    uint8_t* changed;      /* [N] out, may be NULL: 1 if the map changed (stats were recomputed) */
    int32_t* status;       /* [1] device error word, may be NULL.  bit0 (1) an action was out of range;
                              bit1 (2) minecraft_3D_maze: the reference would raise IndexError on this map
                              (helper_3D.py:531, a recorded x or y >= depth); bit2 (4) a search workspace
                              overflowed; bit3 (8) sokoban: more crates than a packed solver state holds (15);
                              bit4 (16) a stat did not fit cfg.record_stat_bytes in the packed record;
                              bit5 (32) pcgrl_step_host: a chunk's results waited more than two seconds for the
                              search kernel (progressive host pipeline) -- the outputs of that step are invalid */
    void*    scratch;      /* pcgrl_scratch_bytes() bytes, may be NULL when that returns 0.  Must be zero-filled
                              once before its first use (it holds hash-table generation counters, solver job
                              lists and, for smb, 4 bytes per env of playthrough-length history, which is why
                              the size depends on n_envs) and must not be shared by launches that can run
                              concurrently */
    uint8_t* static_mask;  /* [N, row_stride] or NULL (ABI 3): StaticTileRepresentation.static_tiles over the map
                              cells (the always-frozen border is implicit).  A frozen cell keeps its tile: the
                              edit is undone, yet still counted as a change (envs/reps/wrappers.py:358-376).
                              Written by random resets when cfg.static_prob / n_static_walls ask for it; with
                              caller-supplied src_grids it is left as the caller set it */
    int32_t* holes;        /* [N, 4] (ABI 4), holey problems only, else NULL: (entrance_y, entrance_x, exit_y, exit_x)
                              in BORDERED coordinates, i.e. the reference's entrance_coords / exit_coords
                              (holey_prob.py:41-42).  Read by step; written by reset per cfg.hole_mode.
                              3D holey problems: [N, 6] = (ez, ey, ex, xz, xy, xx), the FOOT tiles of the entrance and
                              the exit; the head tile is the one above (holey_prob_3D.py:72-92) */
    uint8_t* records;      /* [N, pcgrl_record_stride(cfg)] (ABI 5) or NULL: one packed result record per env, what
                              step() returns besides the observation (pcgrl_env.py:329-342: reward, done, info stats):
                                offset 0            float32 reward
                                offset 4            n_stats values of cfg.record_stat_bytes each (the env's CURRENT stats)
                                offset stride - 2   uint8 done, uint8 changed
                              written by step next to reward / done / stats (which stay the int32 view of the same
                              values); resets refresh the stats part only.  One contiguous device range per env range,
                              so a host step needs ONE device-to-host copy (pcgrl_step_host_packed) */
    int32_t* worklist;     /* [pcgrl_worklist_ints(cfg, N)] int32 (ABI 5) or NULL, zero-filled once before its first
                              use and not shared by concurrent launches: scratch of the SPLIT step path of the
                              bit-board problems (binary, zelda, binary_holey; not the cellular representation) --
                              pcgrl_step then runs three kernels (representation update + global list of changed
                              envs; stat searches with every lane busy; reward / outputs) instead of the fused one.
                              NULL: the fused single-kernel path.  Results are identical either way */
    uint8_t* cache;        /* [N, pcgrl_cache_stride(cfg)] (ABI 5) or NULL; only with worklist, and only where
                              pcgrl_cache_stride(cfg) > 0 (binary, maps up to 16x16, one-cell actions): per-env
                              search state (passable bit-board, one far tile per component, a cell of a longest-path
                              component) that lets step recompute regions / path-length INCREMENTALLY around the
                              edited cell.  Written by reset and by every step; derived state, bit-identical stats.
                              The grids of a shard with a cache must only change through pcgrl_step / pcgrl_reset */
} pcgrl_state;

/* -- queries (host only, no CUDA calls) ------------------------------------------------------- */
int32_t     pcgrl_abi_version(void);
const char* pcgrl_last_error(void);
/* Validate a config and fill derived fields left at 0 (row_stride). */
int32_t     pcgrl_config_check(pcgrl_config* cfg);
int64_t     pcgrl_scratch_bytes(const pcgrl_config* cfg, int64_t n_envs);
/* Algorithmic HBM bytes one env-step moves (SURVEY.md 8d: 2G + A + 8K + 5 [+ 16K per-env targets]). */
int64_t     pcgrl_step_bytes(const pcgrl_config* cfg);

/* Bytes per env of pcgrl_state.records: 4 + n_stats * record_stat_bytes + 2 rounded up to a multiple of 4
 * (0 when cfg.record_stat_bytes == 0). */
int32_t     pcgrl_record_stride(const pcgrl_config* cfg);

/* Sizes of pcgrl_state.worklist (in int32 elements; 0 = this config has no split path) and of one env's row
 * of pcgrl_state.cache (bytes; 0 = no incremental search for this config). */
int64_t     pcgrl_worklist_ints(const pcgrl_config* cfg, int64_t n_envs);
int32_t     pcgrl_cache_stride(const pcgrl_config* cfg);

/* -- launches ---------------------------------------------------------------------------------- */
/* One env-step for every env of the shard.  `actions` layout depends on cfg->action_kind. */
int32_t pcgrl_step(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions, void* stream);

/* Representation.update for every env (envs/reps/*.py update; what evo/evolve.py:1082-1085 calls): map edit,
 * pos / n_step advance, changed[N] = the reference's `change`. No stats, reward, counters or done.
 * Takes the same `actions` as pcgrl_step and sets status bit 0 for an invalid action as it does.  Writes only
 * grids, pos, n_step, changed and status (reads static_mask when set); needs grids, pos, n_step and changed, and
 * no holes for a holey problem.  One launch.  Afterwards `stats` no longer describe the maps (evolution calls
 * pcgrl_stats / pcgrl_stats_holey at the end of the episode), and the search cache of a shard that has one
 * (pcgrl_state.cache) no longer describes its grids: such a shard needs pcgrl_reset before its next pcgrl_step. */
int32_t pcgrl_update(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions, void* stream);

/* (Re)start episodes: PcgrlEnv.reset (envs/pcgrl_env.py:158-188) + Representation.reset
 * (envs/reps/representation.py:65-76) + ControlWrapper.reset (control_wrappers.py:174-187).
 *   mask      [N] uint8 or NULL (= all envs): which envs to reset
 *   src_grids [N, row_stride] int8 or NULL: initial maps (set_map, pcgrl_ctrl_env.py:12-14); NULL = draw
 *             each cell from the tile distribution with Philox4x32-10 keyed by (seed, env, epoch)
 *   src_pos   [N, 3] int32 or NULL: start positions (turtle); NULL = narrow: cell 0, turtle: random
 * Zeroes the counters and recomputes stats; reward/done keep what the last step wrote (so an auto-reset
 * does not erase the finishing step's outputs). */
int32_t pcgrl_reset(const pcgrl_config* cfg, const pcgrl_state* st, const uint8_t* mask,
                    const int8_t* src_grids, const int32_t* src_pos, uint64_t seed, uint64_t epoch,
                    void* stream);

/* Stats only: Problem.get_stats on n grids (evolution's terminal call, evo/evolve.py:1107-1116).
 * grids [n, row_stride] int8 -> stats [n, K] int32. */
int32_t pcgrl_stats(const pcgrl_config* cfg, const int8_t* grids, int32_t* stats, int64_t n, void* scratch,
                    void* stream);
/* Same for a holey problem: holes [n, 4] int32 as in pcgrl_state.holes (BinaryHoleyProblem.get_stats reads
 * self.entrance_coords / self.exit_coords, binary_holey_prob.py:62-63); [n, 6] for minecraft_3D_dungeon_holey; [n, 7]
 * for minecraft_3D_holey_maze: the six coordinates and the path length the previous get_stats call on the same
 * problem object found (reported as this call's path-length, minecraft_3D_holey_maze_prob.py:92-93; 0 at first). */
int32_t pcgrl_stats_holey(const pcgrl_config* cfg, const int8_t* grids, const int32_t* holes, int32_t* stats,
                          int64_t n, void* scratch, void* stream);

/* Observation tensors (control_pcgrl/wrappers.py Cropped :407-437 + OneHotEncoding :232-257 + ToImage
 * :140-150, and ControlWrapper.observe_metric_trgs control_wrappers.py:189-214).
 *   crop != 0 : window obs_dims centred on pos, channel 0 = out-of-bounds, C+1 one-hot channels
 *   crop == 0 : the whole map, C one-hot channels (wide / cellular stacks)
 *   n_ctrl controlled metrics prepend 2*n_ctrl constant planes (trg/range, value/range); ctrl_idx[i] is the
 *   stat index, ctrl_range[i] = |hi - lo| of cond_bounds.
 *   out_kind: 0 = uint8, 1 = float32, 2 = float64 (the reference's np.eye dtype), 3 = uint8 TILE CODES instead of
 *   one-hot records (Cropped's own output, the input of OneHotEncoding: 0 = out of bounds, tile t -> t + 1 behind a
 *   crop; for policies that embed the tile themselves -- a third of the bytes; no target planes).
 *   Output layout [N, *obs_dims, channels] (channels last):
 *   [2*n_ctrl target planes | C+1 or C one-hot | static_builds]. */
typedef struct pcgrl_obs_args {
    int32_t crop;
    int32_t obs_dims[3];
    int32_t n_ctrl;
    int32_t ctrl_idx[PCGRL_MAX_STATS];
    double  ctrl_range[PCGRL_MAX_STATS];
    int32_t out_kind;
    void*   out;
    int32_t static_channel;   /* ABI 3, crop only: append the 'static_builds' plane after the one-hot channels
                                 (wrappers.py:451-453): the BORDERED frozen-tile mask cropped with the map's
                                 padding, i.e. sampled one cell up-left of the map channels (border = 1) */
    int32_t holey_border_tile;/* ABI 4, holey problems only (else ignored): the observed map is the BORDERED map
                                 (dims + 2: border cells show this tile, the two holes of pcgrl_state.holes the empty
                                 tile 0) and positions are shifted by one, as HoleyRepresentation.get_observation
                                 returns it (envs/reps/wrappers.py:153-160); obs_dims are then the window + 2 (crop) or
                                 the map dims + 2 (no crop), :162-174 */
} pcgrl_obs_args;
int32_t pcgrl_observe(const pcgrl_config* cfg, const pcgrl_state* st, const pcgrl_obs_args* obs, void* stream);

/* -- host-buffer convenience (the end-to-end path timed as `e2e` in bench.py) ------------------ */
/* Copies `actions` (host, pinned or pageable) to `actions_dev`, runs pcgrl_step, copies reward/done/stats
 * back to the host buffers, and synchronises the stream.  Any host pointer may be NULL to skip that copy. */
int32_t pcgrl_step_host(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions_host,
                        void* actions_dev, int64_t action_bytes, float* reward_host, uint8_t* done_host,
                        int32_t* stats_host, void* stream);

/* Same with compact host I/O (ABI 5): the ONLY device-to-host traffic is pcgrl_state.records -> records_host
 * ([N, pcgrl_record_stride] bytes, one copy per pipeline chunk instead of three); actions may use
 * cfg.action_elem_bytes = 1 / 2.  st->records must be set. */
int32_t pcgrl_step_host_packed(const pcgrl_config* cfg, const pcgrl_state* st, const void* actions_host,
                               void* actions_dev, int64_t action_bytes, void* records_host, void* stream);

/* Counter of kernels this library has launched in this process (for bench.py's gpu_launches). */
int64_t pcgrl_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PCGRL_B200_H */
