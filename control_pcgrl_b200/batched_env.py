"""BatchedPcgrlEnv: N PCGRL level grids stepped at once on one B200.

Host-side mirror of the reference's env step for a whole batch:
  PcgrlEnv.reset/step           control_pcgrl/envs/pcgrl_env.py:158-188, 267-342
  Representation.update         control_pcgrl/envs/reps/{narrow,turtle,wide,ca}_rep.py
  Problem.get_stats             control_pcgrl/envs/probs/<game>/*_prob.py
  ControlWrapper reward/targets control_pcgrl/control_wrappers.py:174-244, 318-345
  obs wrappers                  control_pcgrl/wrappers.py:140-150, 232-257, 407-437

All state lives in HBM as torch tensors; every method launches the hand-written sm_100a kernels of
libpcgrl_sm100.so through the C ABI (include/pcgrl_b200.h).  PyTorch is only the allocator / stream
provider.  No CPU path exists: constructing this class without CUDA raises.
"""
from __future__ import annotations

import contextlib
import math
from collections import OrderedDict
from types import SimpleNamespace

import numpy as np
import torch

from . import _lib
from .config import normalise
from .problems import HOLEY_PROBLEMS, REPRESENTATION_ALIASES, get_spec


def _ptr(t):
    return None if t is None else t.data_ptr()


_NULL_CTX = contextlib.nullcontext()


class BatchedPcgrlEnv:
    def __init__(self, cfg, n_envs: int, device="cuda:0", env_offset: int = 0, seed: int = 0,
                 action_kind: str | None = None, auto_reset: bool = False, random_init_probs: bool = True,
                 reward_mode: str = "control", compact_host_io: bool = False, split_step: bool = True,
                 n_agents: int | None = None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.PcgrlError("control_pcgrl_b200 needs a CUDA device (there is no CPU fallback)")
        c = normalise(cfg)
        self.cfg = cfg
        self.problem = c.problem
        self.representation = REPRESENTATION_ALIASES[c.representation]
        self.map_shape = c.map_shape
        self.obs_window = c.obs_window
        self.spec = get_spec(self.problem, self.map_shape)
        self.n_envs = int(n_envs)
        self.device = torch.device(device)
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.env_offset = int(env_offset)
        self.seed = int(seed)
        self.auto_reset = auto_reset
        self.ndim = len(self.map_shape)
        self.cells = int(np.prod(self.map_shape))
        self.row_stride = (self.cells + 15) // 16 * 16
        self.n_tiles = self.spec.n_tiles
        self.stat_names = list(self.spec.stat_names)
        self.K = len(self.stat_names)

        # pcgrl_env.py:235-241
        self.max_iterations = self.cells * c.max_board_scans + 1
        self.max_changes = None if c.change_percentage is None else max(int(c.change_percentage * self.cells), 1)

        # ControlWrapper.__init__ (control_wrappers.py:27-121)
        self.ctrl_metrics = list(c.controls or [])
        self.static_trgs = OrderedDict(self.spec.static_trgs)
        self.cond_bounds = dict(self.spec.cond_bounds)
        self.metric_weights = {k: 0 for k in self.spec.reward_weights}
        self.metric_weights.update(c.weights)
        self.all_metrics = list(self.ctrl_metrics) + [k for k in self.static_trgs if k not in self.ctrl_metrics]
        self.param_ranges = {k: abs(self.cond_bounds[k][1] - self.cond_bounds[k][0]) for k in self.ctrl_metrics}

        rep = self.representation
        # multi-agent (cfg.multiagent.n_agents; envs/reps/wrappers.py:612-651 MultiAgentTurtleRepresentation,
        # wrappers.py:697-736 MultiAgentWrapper): every agent keeps its own turtle position on the shared map, and a
        # multi-agent step is one full env step per agent, in agent order.  0 / 1 = the single-agent env.
        self.n_agents = int(c.n_agents if n_agents is None else n_agents)
        if self.n_agents > 1 and rep != "turtle":
            raise ValueError("multi-agent envs need the turtle representation (upstream, MultiAgentNarrowRepresentation "
                             "raises 'Busted for now', envs/reps/wrappers.py:669)")
        # ShowAgentRepresentation (cfg.show_agents, envs/reps/wrappers.py:189-232): an 'agent_occupancy' plane behind
        # the map channels of every agent's observation; upstream it needs several agents (:207-208)
        self.show_agents = bool(c.show_agents) and self.n_agents > 1
        # representation wrappers (envs/reps/wrappers.py wrap_rep :717-722)
        self.act_window = c.act_window
        if self.act_window is not None:
            # MultiActionRepresentation only runs on the narrow rep upstream (turtle has no n_step, wide no _pos)
            if rep != "narrow":
                raise ValueError("act_window (MultiActionRepresentation) is only supported on the narrow representation")
            if len(self.act_window) != self.ndim:
                raise ValueError("act_window must have one entry per map axis (wrappers.py:425-426)")
            if action_kind not in (None, "patch"):
                raise ValueError("act_window needs action_kind 'patch'")
            action_kind = "patch"
        self.static_tile_wrapper = c.static_tile_wrapper
        if self.static_tile_wrapper and rep not in ("narrow", "turtle"):
            raise ValueError("static_tile_wrapper (StaticTileRepresentation) only runs on narrow / turtle upstream")
        self.static_prob = float(c.static_prob or 0)
        self.n_static_walls = int(c.n_static_walls or 0)
        self._static_eval_mode = False
        if action_kind is None:
            action_kind = {"narrow": "int32", "turtle": "int32", "wide": "wide_flat", "cellular": "ca_logits"}[rep]
        self.action_kind = action_kind
        ak = {"int32": _lib.ACT_INT32, "wide_coords": _lib.ACT_WIDE_COORDS, "wide_flat": _lib.ACT_WIDE_FLAT,
              "ca_tiles": _lib.ACT_CA_TILES, "ca_logits": _lib.ACT_CA_LOGITS, "patch": _lib.ACT_PATCH}[action_kind]

        cc = _lib.Config()
        cc.abi_version = _lib.PCGRL_ABI_VERSION
        cc.problem = _lib.PROB_IDS[self.problem]
        cc.representation = _lib.REP_IDS[rep]
        cc.action_kind = ak
        cc.ndim = self.ndim
        for i in range(3):
            cc.dims[i] = self.map_shape[i] if i < self.ndim else 1
        cc.n_tiles = self.n_tiles
        cc.n_stats = self.K
        cc.row_stride = self.row_stride
        cc.max_iterations = int(math.floor(self.max_iterations))
        cc.max_changes = -1 if self.max_changes is None else int(self.max_changes)
        # ActionMap takes (h, w) from the observation space == obs_window (wrappers.py:283-287, SURVEY A-7)
        cc.act_h, cc.act_w = (self.obs_window[0], self.obs_window[1]) if ak == _lib.ACT_WIDE_FLAT else (0, 0)
        cc.targets_per_env = 1 if self.ctrl_metrics else 0
        if action_kind == "patch":
            for i in range(3):
                cc.act_window[i] = self.act_window[i] if i < self.ndim else 1
        if self.static_tile_wrapper:
            cc.static_prob = self.static_prob
            cc.n_static_walls = self.n_static_walls
            cc.wall_tile = 1          # Problem._wall_tile = tiles[1] (envs/probs/problem.py:41)
        # holey problems (envs/pcgrl_holey_env.py, envs/probs/holey_prob.py): entrance / exit per env
        self.holey = self.problem in HOLEY_PROBLEMS
        self.fixed_holes = bool(c.fixed_holes)
        cc.hole_mode = (_lib.HOLES_FIXED if self.fixed_holes else _lib.HOLES_RANDOM) if self.holey else _lib.HOLES_GIVEN
        cc.init_random_probs = 1 if random_init_probs else 0
        # "control": ControlWrapper's loss delta (what step() pays at this commit); "range": the legacy
        # Problem.get_reward sum of get_range_reward terms (helper.py:550-560), bands in `targets`
        if reward_mode not in ("control", "range"):
            raise ValueError(f"reward_mode {reward_mode!r}")
        if reward_mode == "range" and not self.spec.range_bands:
            raise ValueError(f"the reference defines no legacy get_reward for {self.problem}")
        self.reward_mode = reward_mode
        cc.reward_mode = _lib.REWARD_RANGE if reward_mode == "range" else _lib.REWARD_CONTROL
        # compact host I/O (ABI 5): scalar actions in the narrowest unsigned type that holds the action space, and
        # one packed result record per env (reward f32 | stats u8 / i16 / i32 | done | changed) so a host step is
        # ONE device-to-host copy per pipeline chunk
        self.compact_host_io = bool(compact_host_io)
        self._act_elem = 4
        self._rec_sb = 0
        if self.compact_host_io:
            if action_kind in ("int32", "wide_flat"):
                n_act = {"narrow": self.n_tiles, "turtle": 4 + self.n_tiles}.get(
                    rep, self.obs_window[0] * self.obs_window[1] * self.n_tiles)
                self._act_elem = 1 if n_act <= 256 else 2 if n_act <= 65536 else 4
            self._rec_sb = self._stat_bytes()
        cc.action_elem_bytes = self._act_elem
        cc.record_stat_bytes = self._rec_sb
        for i, pr in enumerate(self.spec.init_probs):
            cc.init_probs[i] = pr
        for k, name in enumerate(self.stat_names):
            if reward_mode == "range":
                cc.weights[k] = float(self.spec.range_weights.get(name, 0)) if name in self.spec.range_bands else 0.0
            else:
                cc.weights[k] = float(self.metric_weights.get(name, 0)) if name in self.all_metrics else 0.0
        _lib.check(self.lib.pcgrl_config_check(cc), "pcgrl_config_check")
        self._cc = cc

        N, dev = self.n_envs, self.device
        self.grids = torch.zeros((N, self.row_stride), dtype=torch.int8, device=dev)
        # agent_pos[a] is agent a's position tensor; a step / observation of agent a hands its pointer to the kernels
        # as pcgrl_state.pos, so the single-agent layout (and every kernel) is unchanged
        self.agent_pos = torch.zeros((max(self.n_agents, 1), N, 3), dtype=torch.int32, device=dev)
        self.pos = self.agent_pos[0]
        self.n_step = torch.zeros(N, dtype=torch.int32, device=dev)
        self.iteration = torch.zeros(N, dtype=torch.int32, device=dev)
        self.changes = torch.zeros(N, dtype=torch.int32, device=dev)
        self.stats = torch.zeros((N, self.K), dtype=torch.int32, device=dev)
        self.targets = torch.zeros((N if self.ctrl_metrics else 1, self.K, 2), dtype=torch.float64, device=dev)
        self.reward = torch.zeros(N, dtype=torch.float32, device=dev)
        self.done = torch.zeros(N, dtype=torch.uint8, device=dev)
        self.changed = torch.zeros(N, dtype=torch.uint8, device=dev)
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        # StaticTileRepresentation.static_tiles over the map cells (border implicit), envs/reps/wrappers.py:277
        self.static_mask = torch.zeros((N, self.row_stride), dtype=torch.uint8, device=dev) \
            if self.static_tile_wrapper else None
        # (entrance_y, entrance_x, exit_y, exit_x) in bordered coordinates (holey_prob.py:41-42)
        # 3D holey problems: (ez, ey, ex, xz, xy, xx), the foot tiles (holey_prob_3D.py:72-92; the head is the tile above)
        self.hole_ints = 6 if self.ndim == 3 else 4
        self.holes = torch.zeros((N, self.hole_ints), dtype=torch.int32, device=dev) if self.holey else None
        self.record_stride = int(self.lib.pcgrl_record_stride(cc)) if self._rec_sb else 0
        self.records = torch.zeros((N, self.record_stride), dtype=torch.uint8, device=dev) if self._rec_sb else None
        # split step path of the bit-board problems (csrc/step_split.cu): a global work list of changed envs, and
        # for binary maps up to 16x16 the per-env search cache of the incremental stats.  split_step=False keeps the
        # fused single-kernel path; the results are identical (tests/test_gpu_split.py)
        n_wl = int(self.lib.pcgrl_worklist_ints(cc, N)) if split_step else 0
        self.worklist = torch.zeros(n_wl, dtype=torch.int32, device=dev) if n_wl > 0 else None
        self.cache_stride = int(self.lib.pcgrl_cache_stride(cc)) if n_wl > 0 else 0
        self.cache = torch.zeros((N, self.cache_stride), dtype=torch.uint8, device=dev) if self.cache_stride > 0 else None
        nscratch = self.lib.pcgrl_scratch_bytes(cc, N)
        # zero-initialised once: the solver kernels keep generation counters for their hash tables in it
        self.scratch = torch.zeros(int(nscratch), dtype=torch.uint8, device=dev) if nscratch > 0 else None
        self._hio = None
        self._pinned = {}
        self._epoch = 0
        self._synced_steps = None     # steps since the last full reset while all envs are in lock-step
        # set by update(): stats (and the search cache) no longer describe the maps until the next full reset
        self._stats_stale = False
        self.metric_trgs = OrderedDict(self.static_trgs)
        self._write_targets(self.metric_trgs)

        st = _lib.State()
        st.n_envs, st.env_offset = N, self.env_offset
        st.grids, st.pos, st.n_step = _ptr(self.grids), _ptr(self.pos), _ptr(self.n_step)
        st.iteration, st.changes, st.stats = _ptr(self.iteration), _ptr(self.changes), _ptr(self.stats)
        st.targets, st.reward, st.done = _ptr(self.targets), _ptr(self.reward), _ptr(self.done)
        st.changed, st.status, st.scratch = _ptr(self.changed), _ptr(self.status), _ptr(self.scratch)
        st.static_mask = _ptr(self.static_mask)
        st.holes = _ptr(self.holes)
        st.records = _ptr(self.records)
        st.worklist = _ptr(self.worklist)
        st.cache = _ptr(self.cache)
        self._st = st
        self._st_agents = [st]
        for a in range(1, self.n_agents):
            sa = _lib.State.from_buffer_copy(st)
            sa.pos = self.agent_pos[a].data_ptr()
            self._st_agents.append(sa)

    def _stat_bytes(self):
        """Narrowest record type that holds every stat of this problem.  binary family: region counts and path
        lengths, bounded by cond_bounds (binary_prob.py:66-84: 128 / 136 for 16x16), never negative -> uint8 when
        those fit; everything else: the largest of |cond_bounds|, the cell count (tile counts) and the solver
        defaults (sokoban dist-win = W*H*(W+H), sokoban_prob.py:170) -> int16, else int32.  A value that still does
        not fit raises through status bit 4."""
        bound = max([abs(float(v)) for b in self.cond_bounds.values() for v in b] or [0.0])
        if self.problem in ("binary", "binary_holey", "minecraft_2D_maze"):
            if max(bound, math.ceil(self.cells / 2)) <= 255:
                return 1
        hi = max(bound, self.cells * (sum(self.map_shape) if self.problem in ("sokoban", "smb") else 1))
        return 2 if hi <= 32767 else 4

    def record_dtype(self):
        """numpy structured dtype of one packed result record (pcgrl_state.records)."""
        st = {1: np.uint8, 2: np.int16, 4: np.int32}[self._rec_sb]
        return np.dtype({"names": ["reward", "stats", "done", "changed"],
                         "formats": [np.float32, (st, (self.K,)), np.uint8, np.uint8],
                         "offsets": [0, 4, self.record_stride - 2, self.record_stride - 1],
                         "itemsize": self.record_stride})

    # ------------------------------------------------------------------ targets
    def _target_rows(self, trgs):
        if self.reward_mode == "range":
            return np.array([self.spec.range_bands.get(name, (0.0, 0.0)) for name in self.stat_names], dtype=np.float64)
        rows = np.full((self.K, 2), np.nan, dtype=np.float64)
        for k, name in enumerate(self.stat_names):
            t = trgs.get(name, self.static_trgs.get(name, 0))
            if isinstance(t, tuple):
                rows[k] = (float(t[0]), float(t[1]))
            else:
                rows[k, 0] = float(t)
        return rows

    def _write_targets(self, trgs):
        rows = torch.from_numpy(self._target_rows(trgs)).to(self.device)
        self.targets[:] = rows.unsqueeze(0)

    def set_trgs(self, trgs: dict, env_ids=None):
        """ControlWrapper.do_set_trgs (control_wrappers.py:170-172) for all envs or a subset: the targets named in
        `trgs` change IMMEDIATELY, i.e. the next step's reward is loss(new stats) - loss(old stats) under the new
        targets; every other metric's target (static, sampled or set earlier, per env) is left alone.  The
        reference's queueing set_trgs (applied at the next reset, :167-168, 174-178) lives in the single-env
        ControlWrapper facade (envs.py), which calls this at reset time.
        Values: scalars, (lo, hi) tuples (np.arange(lo, hi), hi excluded), or per-env arrays of scalars."""
        idx = slice(None) if env_ids is None else env_ids
        for k, v in trgs.items():
            if k not in self.stat_names:
                raise KeyError(f"unknown metric {k!r} (stats: {self.stat_names})")
            col = self.stat_names.index(k)
            scalar = isinstance(v, tuple) or np.ndim(v) == 0
            if (not scalar or env_ids is not None) and not self.ctrl_metrics:
                raise ValueError("per-env targets need controls (cfg.controls) so targets are stored per env")
            if scalar and env_ids is None:
                self.metric_trgs[k] = v
            if isinstance(v, tuple):
                self.targets[idx, col, 0] = float(v[0])
                self.targets[idx, col, 1] = float(v[1])
            else:
                vals = float(v) if scalar else torch.as_tensor(np.asarray(v, dtype=np.float64), device=self.device)
                self.targets[idx, col, 0] = vals
                self.targets[idx, col, 1] = float("nan")

    do_set_trgs = set_trgs

    def sample_uniform_targets(self, generator=None):
        """The intended UniformNoiseyTargets behaviour (control_wrappers.py:452-458, SURVEY A-25):
        trg_k ~ U(lo_k, hi_k) per env for every controlled metric."""
        for k in self.ctrl_metrics:
            lo, hi = self.cond_bounds[k]
            u = torch.rand(self.n_envs, dtype=torch.float64, device=self.device, generator=generator)
            col = self.stat_names.index(k)
            self.targets[:, col, 0] = u * (hi - lo) + lo
            self.targets[:, col, 1] = float("nan")

    # ------------------------------------------------------------------ views
    @property
    def maps(self):
        """[N, *map_shape] int8 view of the level grids (PcgrlEnv._rep._map for every env)."""
        return self.grids[:, :self.cells].view(self.n_envs, *self.map_shape)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _on_device(self):
        """The C ABI launches on the calling thread's CURRENT CUDA device: make that the env's device for the call
        (a no-op context when it already is -- the common case, and this sits on the per-step path)."""
        if torch.cuda.current_device() == self._dev_index:
            return _NULL_CTX
        return torch.cuda.device(self.device)

    def _pack_grids(self, grids):
        g = torch.as_tensor(np.asarray(grids) if not torch.is_tensor(grids) else grids)
        g = g.to(device=self.device, dtype=torch.int8).reshape(self.n_envs, self.cells)
        if self.row_stride == self.cells:
            return g.contiguous()
        out = torch.zeros((self.n_envs, self.row_stride), dtype=torch.int8, device=self.device)
        out[:, :self.cells] = g
        return out

    # ------------------------------------------------------------------ reset / step
    # StaticTileRepresentation's setters (envs/reps/wrappers.py:268-275, used by rl/evaluate.py:128-129)
    def set_eval_mode(self, eval_mode: bool):
        self._static_eval_mode = bool(eval_mode)
        self._cc.static_eval_mode = 1 if eval_mode else 0

    def set_static_prob(self, static_prob):
        self.static_prob = float(static_prob or 0)
        self._cc.static_prob = self.static_prob

    def set_n_static_walls(self, n_static_walls):
        self.n_static_walls = int(n_static_walls or 0)
        self._cc.n_static_walls = self.n_static_walls

    @property
    def static_tiles(self):
        """[N, *map_shape] uint8 view of the frozen-tile masks (interior of StaticTileRepresentation.static_tiles)."""
        if self.static_mask is None:
            return None
        return self.static_mask[:, :self.cells].view(self.n_envs, *self.map_shape)

    def reset(self, grids=None, pos=None, mask=None, static_tiles=None, holes=None):
        """Start episodes (all envs, or those where mask != 0).  grids: [N,*map_shape] initial maps
        (PcgrlCtrlEnv.set_map semantics) or None for random maps; pos: [N,ndim] start positions;
        static_tiles: [N,*map_shape] frozen-tile masks to use (with static_tile_wrapper; random resets draw
        their own from static_prob / n_static_walls); holes: [N,4] (entrance_y, entrance_x, exit_y, exit_x) in
        bordered coordinates for a holey problem (the reference's _hole_queue, holey_prob.py:43-44), else the
        kernel draws them (or uses the fixed pair with cfg.fixed_holes)."""
        src = self._pack_grids(grids) if grids is not None else None
        cc = self._cc
        if holes is not None:
            if not self.holey:
                raise ValueError("holes are only meaningful for a holey problem")
            hv = torch.as_tensor(np.asarray(holes) if not torch.is_tensor(holes) else holes)
            hv = hv.to(self.device, torch.int32).reshape(self.n_envs, self.hole_ints)
            if mask is None:
                self.holes.copy_(hv)
            else:
                sel = mask.to(self.device).bool()
                self.holes[sel] = hv[sel]
            cc = _lib.Config.from_buffer_copy(self._cc)
            cc.hole_mode = _lib.HOLES_GIVEN
        if static_tiles is not None:
            if self.static_mask is None:
                raise ValueError("static_tiles needs cfg.static_tile_wrapper")
            sm = torch.as_tensor(np.asarray(static_tiles) if not torch.is_tensor(static_tiles) else static_tiles)
            sm = (sm.to(self.device) != 0).to(torch.uint8).reshape(self.n_envs, self.cells)
            if mask is None:
                self.static_mask[:, :self.cells] = sm
            else:
                sel = mask.to(self.device).bool()
                self.static_mask[sel, :self.cells] = sm[sel]
        sp = None
        agent_sp = None
        if pos is not None:
            p = torch.as_tensor(np.asarray(pos) if not torch.is_tensor(pos) else pos).to(self.device, torch.int32)
            if self.n_agents > 1:      # [N, n_agents, ndim]: every agent's spawn position
                agent_sp = torch.zeros((self.n_agents, self.n_envs, 3), dtype=torch.int32, device=self.device)
                agent_sp[:, :, :self.ndim] = p.reshape(self.n_envs, self.n_agents, self.ndim).permute(1, 0, 2)
                p = agent_sp[0, :, :self.ndim]
            sp = torch.zeros((self.n_envs, 3), dtype=torch.int32, device=self.device)
            sp[:, :self.ndim] = p.reshape(self.n_envs, self.ndim)
        m = None
        if mask is not None:
            m = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        self._epoch += 1
        with self._on_device():
            _lib.check(self.lib.pcgrl_reset(cc, self._st, _ptr(m), _ptr(src), _ptr(sp), self.seed, self._epoch,
                                            self._stream()), "pcgrl_reset")
        if self.n_agents > 1:
            self._spawn_agents(agent_sp, m)
        self._synced_steps = 0 if mask is None else None
        if mask is None:
            self._stats_stale = False
        return self.stats

    def _spawn_agents(self, given, mask):
        """MultiAgentTurtleRepresentation.reset (envs/reps/wrappers.py:616-627): the agents start on distinct map
        cells drawn without replacement (given: [n_agents, N, 3] explicit positions).  The draw is this env's own
        (torch generator on the device): like every random reset it is outside the parity contract."""
        A, N = self.n_agents, self.n_envs
        if given is None:
            g = torch.Generator(device=self.device).manual_seed((self.seed * 1000003 + self._epoch) & 0x7FFFFFFF)
            picks = []
            for a in range(A):
                free = max(self.cells - a, 1)
                r = torch.randint(0, free, (N,), generator=g, device=self.device)
                if a < self.cells:          # the r-th cell that no earlier agent took
                    prev = torch.sort(torch.stack(picks), dim=0).values if picks else None
                    for q in range(len(picks)):
                        r = r + (r >= prev[q]).to(r.dtype)
                picks.append(r)
            given = torch.zeros((A, N, 3), dtype=torch.int32, device=self.device)
            for a in range(A):
                rem = picks[a]
                for ax in range(self.ndim - 1, -1, -1):
                    given[a, :, ax] = (rem % self.map_shape[ax]).to(torch.int32)
                    rem = rem // self.map_shape[ax]
        if mask is None:
            self.agent_pos.copy_(given)
        else:
            sel = mask.bool()
            self.agent_pos[:, sel] = given[:, sel]

    def _agent_state(self, agent):
        if not 0 <= int(agent) < max(self.n_agents, 1):
            raise IndexError(f"agent {agent} of {max(self.n_agents, 1)}")
        return self._st_agents[int(agent)]

    def step(self, actions: torch.Tensor, agent: int = 0):
        """One env-step for all N envs.  `actions` is a device tensor laid out per `action_kind`.
        Returns (reward[N] f32, done[N] u8) device tensors (overwritten by the next step).
        agent: with n_agents > 1, whose turtle acts (MultiAgentWrapper.step, wrappers.py:724-731, steps the env once
        per agent)."""
        self._check_fresh("step")
        a = self._check_actions(actions)
        with self._on_device():
            _lib.check(self.lib.pcgrl_step(self._cc, self._agent_state(agent), a.data_ptr(), self._stream()),
                       "pcgrl_step")
        if self.n_agents > 1 and self._in_agent_round:
            if self._synced_steps is not None:
                self._synced_steps += 1
        else:
            self._after_step()
        return self.reward, self.done

    _in_agent_round = False

    def update(self, actions: torch.Tensor, agent: int = 0) -> torch.Tensor:
        """Representation.update for all N envs (envs/reps/*.py), the call evolution's generator loop makes at every
        iteration (evo/evolve.py:1082-1085, _get_stats_on_step = False): edits the maps and advances pos / n_step,
        nothing else -- no stats, reward, iteration / changes counters or done.  `actions` as for step() (same layout
        and dtype, including compact_host_io's narrow types); agent: whose turtle acts with n_agents > 1.
        Returns changed[N] u8 (the reference's `change`; overwritten by the next call).

        Afterwards `stats` no longer describe the maps: step(), step_agents(), step_host() and observe() with control
        planes raise until a full reset().  End-of-episode stats: compute_stats(env.maps, holes=env.holes)."""
        a = self._check_actions(actions)
        with self._on_device():
            _lib.check(self.lib.pcgrl_update(self._cc, self._agent_state(agent), a.data_ptr(), self._stream()),
                       "pcgrl_update")
        self._stats_stale = True
        return self.changed

    def _check_fresh(self, what):
        if self._stats_stale:
            raise RuntimeError(f"{what}: update() edited the maps without recomputing stats, so stats (and the step's "
                               "search cache) are stale; call reset() (all envs) before stepping again")

    def step_agents(self, actions: torch.Tensor):
        """One multi-agent step: actions[N, n_agents], agent a acts a-th (MultiAgentWrapper.step,
        wrappers.py:724-731: a full env step per agent, so iteration advances by n_agents).  Returns
        (reward[n_agents, N] f32, done[n_agents, N] u8); with auto_reset, envs restart once every agent of the round
        saw done (the wrapper's done['__all__'])."""
        self._check_fresh("step_agents")
        A = max(self.n_agents, 1)
        if actions.dim() != 2 or tuple(actions.shape) != (self.n_envs, A):
            raise ValueError(f"actions must be [n_envs, n_agents] = {(self.n_envs, A)}")
        rewards = torch.empty((A, self.n_envs), dtype=torch.float32, device=self.device)
        dones = torch.empty((A, self.n_envs), dtype=torch.uint8, device=self.device)
        self._in_agent_round = True
        try:
            for a in range(A):
                r, d = self.step(actions[:, a].contiguous(), agent=a)
                rewards[a].copy_(r)
                dones[a].copy_(d)
        finally:
            self._in_agent_round = False
        if self.auto_reset:
            if self.max_changes is None and self._synced_steps is not None:
                # lock-step: the round's first agent saw done iff its sub-step count exceeded max_iterations
                if self._synced_steps - (A - 1) > self.max_iterations:
                    self.reset()
            else:
                all_done = dones.min(dim=0).values
                if bool(all_done.any()):
                    self.reset(mask=all_done)
        return rewards, dones

    def _after_step(self):
        if self._synced_steps is not None:
            self._synced_steps += 1
        if not self.auto_reset:
            return
        if self.max_changes is None and self._synced_steps is not None:
            # every env hits `iteration > max_iterations` on the same step: no device->host sync needed
            if self._synced_steps > self.max_iterations:
                self.reset()
        else:
            self.reset(mask=self.done)

    def _action_layout(self):
        """(shape, numpy dtype, torch dtype) of one action batch for this env's action_kind."""
        N = self.n_envs
        scalar = {4: (np.int32, torch.int32), 1: (np.uint8, torch.uint8), 2: (np.uint16, torch.uint16)}[self._act_elem]
        return {"int32": ((N,), *scalar), "wide_flat": ((N,), *scalar),
                "wide_coords": ((N, self.ndim + 1), np.int32, torch.int32),
                "ca_tiles": ((N, self.row_stride), np.int8, torch.int8),
                "ca_logits": ((N, self.n_tiles * self.cells), np.float32, torch.float32),
                "patch": ((N, int(np.prod(self.act_window or (1,)))), np.int32, torch.int32)}[self.action_kind]

    def _check_actions(self, actions):
        if not torch.is_tensor(actions) or actions.device != self.device:
            raise TypeError("actions must be a tensor on the env's device (use step_host for host arrays)")
        shape, _, tdt = self._action_layout()
        if actions.dtype != tdt:
            raise TypeError(f"actions dtype {actions.dtype} != {tdt} for action_kind {self.action_kind}")
        if actions.numel() != int(np.prod(shape)):
            raise ValueError(f"actions shape {tuple(actions.shape)} does not match {shape}")
        return actions.reshape(shape).contiguous()

    def action_shape_dtype(self):
        shape, dt, _ = self._action_layout()
        return shape, dt

    def _pinned_buf(self, name, shape, dtype):
        b = self._pinned.get(name)
        if b is None or tuple(b.shape) != tuple(shape) or b.dtype != dtype:
            b = torch.empty(shape, dtype=dtype, pin_memory=True)
            self._pinned[name] = b
        return b

    def host_action_buffer(self, name="actions"):
        """A pinned host tensor of the action layout; fill it and pass it to step_host to skip the staging copy."""
        shape, _, tdt = self._action_layout()
        return torch.empty(shape, dtype=tdt, pin_memory=True) if name is None else self._pinned_buf(name, shape, tdt)

    def _host_io(self):
        """Per-env constants of the host-buffer path, built once: action layout, pinned result buffers and their
        numpy views (step_host runs every ~0.4 ms at the headline size, so it must not rebuild any of this)."""
        h = self._hio
        if h is None:
            shape, dt, tdt = self._action_layout()
            h = SimpleNamespace(shape=shape, dt=dt, tdt=tdt, numel=int(np.prod(shape)), known={})
            h.nbytes = h.numel * np.dtype(dt).itemsize
            h.act_dev = torch.empty(shape, dtype=tdt, device=self.device)
            if self.compact_host_io:
                h.rec = torch.empty((self.n_envs, self.record_stride), dtype=torch.uint8, pin_memory=True)
                v = h.rec.numpy().view(self.record_dtype()).reshape(self.n_envs)
                h.views = (v["reward"], v["done"], v["stats"], v["changed"])
            else:
                h.r = torch.empty(self.n_envs, dtype=torch.float32, pin_memory=True)
                h.d = torch.empty(self.n_envs, dtype=torch.uint8, pin_memory=True)
                h.s = torch.empty((self.n_envs, self.K), dtype=torch.int32, pin_memory=True)
                h.views = (h.r.numpy(), h.d.numpy(), h.s.numpy())
            self._hio = h
        return h

    def step_host(self, actions, want_stats=True, agent: int = 0):
        """End-to-end step with HOST buffers (the call timed as `e2e`): actions are copied H2D from pinned
        memory, the fused kernel runs, reward / done / stats are copied back, and the stream is synchronised.
        Large binary / zelda shards are cut into chunks whose upload, kernel and download overlap on helper
        streams (pcgrl_step_host).  `actions`: numpy array (staged through a pinned buffer) or an already
        pinned torch tensor of the action layout (used in place).
        Returns numpy views of pinned buffers (reward f32[N], done u8[N], stats [N,K] or None), overwritten by the
        next call.  By default these are three dense arrays (stats int32); with compact_host_io they are strided
        views of ONE packed record array (stats uint8 / int16 as the problem's bounds allow, see record_dtype()),
        downloaded with a single copy per pipeline chunk (pcgrl_step_host_packed)."""
        self._check_fresh("step_host")
        h = self._host_io()
        a_ptr = h.known.get(id(actions))
        if a_ptr is None:
            if torch.is_tensor(actions) and actions.device.type == "cpu" and actions.is_pinned() and \
                    actions.dtype == h.tdt and actions.is_contiguous() and actions.numel() == h.numel:
                if len(h.known) < 4096:     # remember validated pinned buffers (and keep them alive)
                    h.known[id(actions)] = (actions, actions.data_ptr())
                a_ptr = actions.data_ptr()
            else:
                a_pin = self._pinned_buf("actions", h.shape, h.tdt)
                a_pin.view(torch.uint8).numpy().view(h.dt).reshape(h.shape)[...] = \
                    np.asarray(actions).astype(h.dt, copy=False).reshape(h.shape)
                a_ptr = a_pin.data_ptr()
        else:
            a_ptr = a_ptr[1]
        with self._on_device():
            if self.compact_host_io:
                rc = self.lib.pcgrl_step_host_packed(self._cc, self._agent_state(agent), a_ptr, h.act_dev.data_ptr(), h.nbytes,
                                                     h.rec.data_ptr(), self._stream())
            else:
                rc = self.lib.pcgrl_step_host(self._cc, self._agent_state(agent), a_ptr, h.act_dev.data_ptr(), h.nbytes,
                                              h.r.data_ptr(), h.d.data_ptr(), h.s.data_ptr() if want_stats else None,
                                              self._stream())
        if rc:
            _lib.check(rc, "pcgrl_step_host")
        self._after_step()
        return h.views[0], h.views[1], (h.views[2] if want_stats else None)

    def host_io_bytes(self, want_stats=True):
        """(h2d, d2h) bytes one step_host call moves over PCIe, counted from the buffers it copies."""
        shape, dt, _ = self._action_layout()
        h2d = int(np.prod(shape)) * np.dtype(dt).itemsize
        if self.compact_host_io:
            return h2d, self.n_envs * self.record_stride
        return h2d, self.n_envs * (4 + 1 + (4 * self.K if want_stats else 0))

    # ------------------------------------------------------------------ stats / observations
    def compute_stats(self, grids, holes=None, prev_path_length=None) -> torch.Tensor:
        """Problem.get_stats for arbitrary grids [n, *map_shape] (evolution's terminal call).  A holey problem also
        needs holes [n, 4] (3D: [n, 6], the foot tiles) -- its get_stats reads entrance_coords / exit_coords.
        minecraft_3D_holey_maze reports as path-length what the PREVIOUS call on the same problem object found
        (minecraft_3D_holey_maze_prob.py:92-93): pass those lengths as prev_path_length [n] (default 0); the
        length this call finds comes back as the stat `_next-path-length`."""
        g = torch.as_tensor(np.asarray(grids) if not torch.is_tensor(grids) else grids)
        n = g.shape[0]
        g = g.to(device=self.device, dtype=torch.int8).reshape(n, self.cells)
        if self.row_stride != self.cells:
            buf = torch.zeros((n, self.row_stride), dtype=torch.int8, device=self.device)
            buf[:, :self.cells] = g
            g = buf
        g = g.contiguous()
        out = torch.empty((n, self.K), dtype=torch.int32, device=self.device)
        if self.holey:
            if holes is None:
                raise ValueError(f"a holey problem needs holes [n, {self.hole_ints}] for compute_stats")
            hv = torch.as_tensor(np.asarray(holes) if not torch.is_tensor(holes) else holes)
            hv = hv.to(self.device, torch.int32).reshape(n, self.hole_ints)
            if self.problem == "minecraft_3D_holey_maze":
                prev = torch.zeros(n, dtype=torch.int32, device=self.device) if prev_path_length is None else \
                    torch.as_tensor(np.asarray(prev_path_length) if not torch.is_tensor(prev_path_length)
                                    else prev_path_length).to(self.device, torch.int32).reshape(n)
                hv = torch.cat([hv, prev[:, None]], dim=1)
            hv = hv.contiguous()
            with self._on_device():
                _lib.check(self.lib.pcgrl_stats_holey(self._cc, g.data_ptr(), hv.data_ptr(), out.data_ptr(), n,
                                                      _ptr(self.scratch), self._stream()), "pcgrl_stats_holey")
            return out
        with self._on_device():
            _lib.check(self.lib.pcgrl_stats(self._cc, g.data_ptr(), out.data_ptr(), n, _ptr(self.scratch),
                                            self._stream()), "pcgrl_stats")
        return out

    def obs_shape(self, onehot: bool = True):
        crop = self.representation in ("narrow", "turtle")
        dims = self.obs_window if crop else self.map_shape
        if self.holey:      # HoleyRepresentation.get_observation_space (envs/reps/wrappers.py:162-174): map + 2
            dims = tuple(d + 2 for d in dims)
        ch = ((self.n_tiles + 1 if crop else self.n_tiles) if onehot else 1) + 2 * len(self.ctrl_metrics)
        ch += 1 if self.static_mask is not None else 0      # 'static_builds' plane (wrappers.py:451-453)
        ch += 1 if self.show_agents else 0                  # 'agent_occupancy' plane
        return (*dims, ch)

    def _agent_occupancy(self, agent, dims, dtype):
        """[N, *dims]: 1 where any agent stands, in agent `agent`'s window (Cropped pads this key with 0)."""
        nd, dev = self.ndim, self.device
        occ = torch.zeros((self.n_envs, *dims), dtype=dtype, device=dev)
        center = self.agent_pos[agent, :, :nd].long()
        half = torch.tensor([d // 2 for d in dims], device=dev)
        lim = torch.tensor(list(dims), device=dev)
        env_idx = torch.arange(self.n_envs, device=dev)
        for b in range(self.n_agents):
            rel = self.agent_pos[b, :, :nd].long() - center + half
            ok = ((rel >= 0) & (rel < lim)).all(dim=1)
            occ[(env_idx[ok],) + tuple(rel[ok, i] for i in range(nd))] = 1
        return occ

    def observe(self, out: torch.Tensor | None = None, dtype=torch.float32, onehot: bool = True, agent: int = 0):
        """The wrapped observation of every env: [N, *obs_dims, channels] (channels last), exactly what
        CroppedImagePCGRLWrapper / ActionMapImagePCGRLWrapper + ControlWrapper return per env.
        onehot=False (uint8 only, no controls): the tile codes of the crop instead of their one-hot records --
        Cropped's own output (wrappers.py:407-437: 0 = out of bounds, tile t -> t + 1), one channel, for policies
        that embed the tile themselves (SURVEY 8f rank 3).
        agent: with n_agents > 1, whose crop (every agent sees the shared map around its own position)."""
        if self.ctrl_metrics:
            self._check_fresh("observe with control planes")
        if not onehot:
            if self.ctrl_metrics or (out is not None and out.dtype != torch.uint8):
                raise ValueError("onehot=False is a uint8 observation without control planes")
            dtype = torch.uint8
        shape = (self.n_envs, *self.obs_shape(onehot))
        final = None
        if self.show_agents:
            # the kernel writes the map (+ target / static) channels; the occupancy plane is appended here (a handful
            # of scatters, one per agent)
            if out is not None and (tuple(out.shape) != shape or not out.is_contiguous()):
                raise ValueError(f"out must be contiguous with shape {shape}")
            final, out = out, None
            if final is not None:
                dtype = final.dtype
            shape = (*shape[:-1], shape[-1] - 1)
        if out is None:
            out = torch.empty(shape, dtype=dtype, device=self.device)
        if tuple(out.shape) != shape or not out.is_contiguous():
            raise ValueError(f"out must be contiguous with shape {shape}")
        crop = self.representation in ("narrow", "turtle")
        oa = _lib.ObsArgs()
        oa.crop = 1 if crop else 0
        dims = self.obs_window if crop else self.map_shape
        if self.holey:
            # the bordered map with the holes, positions + 1 (HoleyRepresentation.get_observation, wrappers.py:153-160)
            dims = tuple(d + 2 for d in dims)
            oa.holey_border_tile = self.spec.tiles.index(self.spec.border_tile)
        for i in range(3):
            oa.obs_dims[i] = dims[i] if i < self.ndim else 1
        oa.n_ctrl = len(self.ctrl_metrics)
        for i, k in enumerate(self.ctrl_metrics):
            oa.ctrl_idx[i] = self.stat_names.index(k)
            oa.ctrl_range[i] = float(self.param_ranges[k])
        oa.out_kind = {torch.uint8: 0, torch.float32: 1, torch.float64: 2}[out.dtype] if onehot else 3
        oa.out = out.data_ptr()
        oa.static_channel = 1 if self.static_mask is not None else 0
        with self._on_device():
            _lib.check(self.lib.pcgrl_observe(self._cc, self._agent_state(agent), oa, self._stream()), "pcgrl_observe")
        if self.show_agents:
            occ = self._agent_occupancy(agent, shape[1:-1], out.dtype)
            if final is None:
                return torch.cat([out, occ[..., None]], dim=-1)
            final[..., :-1] = out
            final[..., -1] = occ
            return final
        return out

    STATUS_BITS = (
        (1, ValueError, "an action outside the action space reached pcgrl_step (ignored on device)"),
        (2, IndexError, "minecraft_3D_maze: the reference raises IndexError on this map (helper_3D.py:531: a recorded "
                        "x or y >= depth); the stats of that env are not meaningful"),
        (4, RuntimeError, "a search workspace overflowed: the stats of at least one env are NOT the reference's "
                          "(parity lost) -- report the map"),
        (8, RuntimeError, "sokoban: a level with more than 15 crates met the solver preconditions; a packed solver "
                          "state holds 15, so its dist-win / sol-length were not computed"),
        (16, OverflowError, "a stat did not fit the packed result record (record_stat_bytes too small)"),
        (32, RuntimeError, "step_host: a chunk's results waited more than two seconds for the search kernel "
                           "(progressive host pipeline); the outputs of that step are invalid"),
    )

    def check_status(self):
        """Raise the error that matches the device status word (include/pcgrl_b200.h, pcgrl_state.status); one D2H
        sync.  Parity-relevant conditions (workspace overflow, crate limit) outrank a bad action."""
        s = int(self.status.item())
        if not s:
            return
        self.status.zero_()
        for bit, exc, msg in sorted(self.STATUS_BITS, key=lambda b: b[0] not in (4, 8, 32)):
            if s & bit:
                raise exc(f"{msg} [status word {s}]")
        raise RuntimeError(f"unknown device status word {s}")

    def step_bytes(self) -> int:
        return int(self.lib.pcgrl_step_bytes(self._cc))

    def stats_dict(self, i: int):
        row = self.stats[i].tolist()
        return OrderedDict(zip(self.stat_names, row))

    _STATE_TENSORS = ("grids", "agent_pos", "n_step", "iteration", "changes", "stats", "targets", "static_mask", "holes",
                      "records", "cache")

    def state_dict(self):
        """Everything needed to reconstruct the env state (SURVEY.md section 5, checkpoint row), including the
        position of the counter-based reset RNG stream (seed, epoch)."""
        sd = {k: getattr(self, k).clone() for k in self._STATE_TENSORS if getattr(self, k) is not None}
        sd["_epoch"] = int(self._epoch)
        sd["seed"] = int(self.seed)
        sd["_synced_steps"] = self._synced_steps
        sd["_stats_stale"] = bool(self._stats_stale)
        return sd

    def load_state_dict(self, sd):
        want = {k for k in self._STATE_TENSORS if getattr(self, k) is not None}
        have = {k for k in sd if k not in ("_epoch", "seed", "_synced_steps", "_stats_stale")}
        if want != have:
            raise KeyError(f"state_dict keys differ: missing {sorted(want - have)}, unexpected {sorted(have - want)}")
        for k in want:
            if tuple(sd[k].shape) != tuple(getattr(self, k).shape) or sd[k].dtype != getattr(self, k).dtype:
                raise ValueError(f"state_dict[{k!r}]: shape / dtype {tuple(sd[k].shape)} {sd[k].dtype} != "
                                 f"{tuple(getattr(self, k).shape)} {getattr(self, k).dtype}")
        for k in want:
            getattr(self, k).copy_(sd[k])
        self._epoch = int(sd.get("_epoch", self._epoch))
        self.seed = int(sd.get("seed", self.seed))
        self._synced_steps = sd.get("_synced_steps")     # lock-step episode clock (None: envs are out of step)
        self._stats_stale = bool(sd.get("_stats_stale", False))    # checkpoints from before update() have no flag
