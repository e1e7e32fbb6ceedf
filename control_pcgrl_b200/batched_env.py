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

    def step(self, actions: torch.Tensor, agent: int = 0, env_ids=None):
        """One env-step for all N envs.  `actions` is a device tensor laid out per `action_kind`.
        Returns (reward[N] f32, done[N] u8) device tensors (overwritten by the next step).
        agent: with n_agents > 1, whose turtle acts (MultiAgentWrapper.step, wrappers.py:724-731, steps the env once
        per agent).
        env_ids: a 1-D integer array / tensor of M DISTINCT env indices (any order): only those envs step, env_ids[j]
        taking row j of `actions` (the step layout with M rows), and every other env keeps its state and its last
        outputs bit for bit (pcgrl_step_envs).  Returns fresh compact (reward[M] f32, done[M] u8).  With auto_reset,
        the listed envs that finished restart.  A bad or repeated index raises IndexError / ValueError before
        anything is launched (a device tensor costs one sort and one sync for that check)."""
        if env_ids is not None:
            return self._step_envs(actions, agent, env_ids)
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

    def _step_envs(self, actions, agent, env_ids):
        self._check_fresh("step")
        rows = self._check_env_ids(env_ids, distinct=True)
        m = rows.numel()
        a = self._check_actions(actions, m)
        st = self._agent_state(agent)
        if m == 0:
            return (torch.empty(0, dtype=torch.float32, device=self.device),
                    torch.empty(0, dtype=torch.uint8, device=self.device))
        work = self._work(int(self.lib.pcgrl_step_envs_work_bytes(self._cc, m)))
        with self._on_device():
            _lib.check(self.lib.pcgrl_step_envs(self._cc, st, a.data_ptr(), rows.data_ptr(), m, work.data_ptr(),
                                                self._stream()), "pcgrl_step_envs")
        idx = rows.long()
        reward, done = self.reward[idx], self.done[idx]
        self._synced_steps = None
        if self.auto_reset:     # the listed envs that finished: unlisted rows of self.done are older steps' flags
            mask = torch.zeros(self.n_envs, dtype=torch.uint8, device=self.device)
            mask[idx] = done
            self.reset(mask=mask)
        return reward, done

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

    # ------------------------------------------------------------------ lookahead
    def lookahead(self, actions: torch.Tensor, env_ids=None, agent: int = 0, obs_dtype=None, onehot: bool = True,
                  obs_out: torch.Tensor | None = None):
        """What step() would return for a list of (env, action) candidates, without stepping.  Candidate j pairs env
        env_ids[j] (j when env_ids is None) with row j of `actions` (the step layout with M rows, M = len(env_ids) or
        n_envs).  Returns fresh device tensors (reward[M] f32, done[M] u8, stats[M, K] i32, changed[M] u8): the
        reward (bit for bit), done, stats row and changed flag that env would get from step() if it took that action
        next.  Indices may come in any order and repeat.  agent: with n_agents > 1, whose turtle would act.
        Nothing of the env changes, except that check_status() then reports what such a step would (an invalid
        action: ValueError); no auto-reset.  A bad env index raises IndexError before anything is launched (a device
        tensor costs one reduction and one sync for that check).
        obs_dtype / obs_out: also return the observation [M, *obs_shape] as a fifth tensor, row j byte for byte what
        observe(dtype=obs_dtype, onehot=onehot, agent=agent) would return for that env right after that step
        (pcgrl_lookahead_obs): target planes from the candidate's new stats, the terminal observation of a candidate
        that would end the episode.  obs_out, a contiguous [M, *obs_shape] tensor, receives it; onehot=False is the
        uint8 tile codes, as for observe()."""
        self._check_fresh("lookahead")
        if obs_dtype is not None and onehot:
            self._check_obs_dtype(obs_dtype)
        rows = None if env_ids is None else self._check_env_ids(env_ids)
        m = self.n_envs if rows is None else rows.numel()
        a = self._check_actions(actions, m)
        K = self.K
        out = (torch.empty(m, dtype=torch.float32, device=self.device), torch.empty(m, dtype=torch.uint8, device=self.device),
               torch.empty((m, K), dtype=torch.int32, device=self.device), torch.empty(m, dtype=torch.uint8, device=self.device))
        if obs_dtype is None and obs_out is None:
            self._lookahead(a, rows, m, agent, *out)
            return out
        return (*out, self._lookahead_obs(a, rows, m, agent, out, obs_out, obs_dtype or torch.float32, onehot))

    def _lookahead(self, a, rows, m, agent, reward, done, stats, changed, obs=None):
        """pcgrl_lookahead, or with `obs` (pcgrl_obs_args) pcgrl_lookahead_obs."""
        if m == 0:
            return
        st = self._agent_state(agent)
        if obs is None:
            work = self._work(int(self.lib.pcgrl_lookahead_work_bytes(self._cc, m)))
            with self._on_device():
                _lib.check(self.lib.pcgrl_lookahead(self._cc, st, a.data_ptr(), _ptr(rows), m, reward.data_ptr(),
                                                    done.data_ptr(), changed.data_ptr(), stats.data_ptr(),
                                                    work.data_ptr(), self._stream()), "pcgrl_lookahead")
            return
        work = self._work(int(self.lib.pcgrl_lookahead_obs_work_bytes(self._cc, m)))
        with self._on_device():
            _lib.check(self.lib.pcgrl_lookahead_obs(self._cc, st, obs, a.data_ptr(), _ptr(rows), m, reward.data_ptr(),
                                                    done.data_ptr(), changed.data_ptr(), stats.data_ptr(),
                                                    work.data_ptr(), self._stream()), "pcgrl_lookahead_obs")

    def _lookahead_obs(self, a, rows, m, agent, outs, obs_out, dtype, onehot):
        """_lookahead with the observation: -> obs [m, *obs_shape]."""
        final, ob, oa = self._obs_buffers(m, obs_out, dtype, onehot)
        self._lookahead(a, rows, m, agent, *outs, obs=oa)
        occ = None
        if self.show_agents:
            ids = torch.arange(m, device=self.device) if rows is None else rows
            occ = self._agent_occupancy(agent, ob.shape[1:-1], ob.dtype, ids, self._turtle_after(a, ids, agent))
        return self._obs_finish(final, ob, occ)

    def _turtle_after(self, a, rows, agent):
        """[M, 3]: where agent `agent`'s turtle stands after action a[j] in env rows[j] (reps/turtle_rep.py:87-107:
        0..3 move along axis 0 / 1, clamped to the map; a write or an invalid action stays).  The library returns no
        positions, and multi-agent envs are turtle-only, so the occupancy plane of a lookahead takes them from here."""
        pos = self.agent_pos[agent][rows.long()].long()
        a = a.reshape(-1).to(torch.int64)
        for axis in (0, 1):
            step = (a == 2 * axis + 1).long() - (a == 2 * axis).long()
            pos[:, axis] = (pos[:, axis] + step).clamp(0, self.map_shape[axis] - 1)
        return pos

    def _work(self, need):
        """The work buffer of lookahead and of step(env_ids=...), at least `need` bytes (both keep the solver scratch at
        the same offset, so one buffer serves both)."""
        if self._la_work is None or self._la_work.numel() < need:
            # zero-filled when allocated: the solver kernels keep generation counters in it
            self._la_work = None
            self._la_work = torch.zeros(need, dtype=torch.uint8, device=self.device)
        return self._la_work

    _la_work = None
    LOOKAHEAD_CHUNK = 1 << 22     # candidates per launch of lookahead_all: bounds the work buffer
    LOOKAHEAD_OBS_CHUNK_BYTES = 1 << 30   # ... and the observation bytes of one launch (and its temporaries)

    def n_discrete_actions(self):
        """Size of the Discrete action space (narrow C, turtle 4 + C, flat wide act_h * act_w * C)."""
        if self.action_kind not in ("int32", "wide_flat"):
            raise ValueError(f"action_kind {self.action_kind!r} is not a Discrete action space")
        return {"narrow": self.n_tiles, "turtle": 4 + self.n_tiles}.get(
            self.representation, self._cc.act_h * self._cc.act_w * self.n_tiles)

    def lookahead_all(self, env_ids=None, agent: int = 0, obs_dtype=None, onehot: bool = True):
        """lookahead() of every action of the Discrete action space for each env of env_ids (default all): returns
        reward [M, A] f32, done [M, A] u8, stats [M, A, K] i32 and changed [M, A] u8, column a being action a.
        Runs in chunks of at most LOOKAHEAD_CHUNK candidates, env-major, without a host sync (env_ids=None).
        Raises ValueError for cellular, patch and wide-coordinate actions, and for flat wide actions whose ActionMap
        (act_h, act_w) reaches past the map: part of that space is actions the reference rejects.
        obs_dtype: also return obs [M, A, *obs_shape], lookahead()'s observation of every candidate; chunks then hold at
        most LOOKAHEAD_OBS_CHUNK_BYTES of it.  Mind the size: it is M * A observations, so wide actions are expensive
        (16 Ki binary-wide envs x 512 actions x 6 KB of float32 crop is about 50 GB; bfloat16 halves that).  It is meant
        for narrow and turtle envs; elsewhere call lookahead() on chosen candidates."""
        self._check_fresh("lookahead_all")
        if obs_dtype is not None and onehot:
            self._check_obs_dtype(obs_dtype)
        A = self.n_discrete_actions()
        if self.action_kind == "wide_flat":
            # action (y, x, v): the write goes to _map[x, y], so x must be a row and y a column (wrappers.py:304-323)
            if self._cc.act_w > self.map_shape[0] or self._cc.act_h > self.map_shape[1]:
                raise ValueError(f"ActionMap ({self._cc.act_h}, {self._cc.act_w}) reaches past the map {self.map_shape}")
        rows = None if env_ids is None else self._check_env_ids(env_ids)
        M = self.n_envs if rows is None else rows.numel()
        dev, K = self.device, self.K
        reward = torch.empty((M, A), dtype=torch.float32, device=dev)
        done = torch.empty((M, A), dtype=torch.uint8, device=dev)
        stats = torch.empty((M, A, K), dtype=torch.int32, device=dev)
        changed = torch.empty((M, A), dtype=torch.uint8, device=dev)
        _, _, tdt = self._action_layout()
        per_cand = self.LOOKAHEAD_CHUNK
        obs = None
        if obs_dtype is not None:
            oshape = self.obs_shape(onehot)
            obs = torch.empty((M, A, *oshape), dtype=obs_dtype if onehot else torch.uint8, device=dev)
            per_cand = max(1, min(per_cand, self.LOOKAHEAD_OBS_CHUNK_BYTES // (math.prod(oshape) * obs.element_size())))
        per = max(1, per_cand // A)
        for lo in range(0, M, per):
            hi = min(M, lo + per)
            c = torch.arange((hi - lo) * A, dtype=torch.int32, device=dev)
            env = c // A + lo if rows is None else rows[lo:hi].repeat_interleave(A, output_size=(hi - lo) * A)
            acts = (c % A).to(tdt)
            env = env.to(torch.int32).contiguous()
            outs = (reward[lo:hi], done[lo:hi], stats[lo:hi], changed[lo:hi])
            if obs is None:
                self._lookahead(acts, env, (hi - lo) * A, agent, *outs)
            else:
                self._lookahead_obs(acts, env, (hi - lo) * A, agent, outs, obs[lo:hi].view(-1, *oshape), obs.dtype,
                                    onehot)
        if obs is None:
            return reward, done, stats, changed
        return reward, done, stats, changed, obs

    def _check_fresh(self, what):
        if self._stats_stale:
            raise RuntimeError(f"{what}: update() edited the maps without recomputing stats, so stats (and the step's "
                               "search cache) are stale; call reset() (all envs) before stepping again")

    # ------------------------------------------------------------------ packed env rows
    _row_layout_cache = None
    _fork_buf = None
    # row_fields name -> (pcgrl_row_layout field, dtype)
    _ROW_FIELDS = (("grids", "grid", torch.int8), ("static_mask", "static_mask", torch.uint8),
                   ("cache", "cache", torch.uint8), ("records", "records", torch.uint8),
                   ("targets", "targets", torch.float64), ("stats", "stats", torch.int32),
                   ("holes", "holes", torch.int32), ("agent_pos", "pos", torch.int32),
                   ("n_step", "n_step", torch.int32), ("iteration", "iteration", torch.int32),
                   ("changes", "changes", torch.int32), ("reward", "reward", torch.float32),
                   ("done", "done", torch.uint8), ("changed", "changed", torch.uint8))

    def _row_layout(self):
        """pcgrl_row_layout of this env's rows, with every agent's position array (agent_pos) in them."""
        if self._row_layout_cache is None:
            lay = _lib.RowLayout()
            _lib.check(self.lib.pcgrl_env_row_layout(self._cc, self._st, self.agent_pos.shape[0], lay),
                       "pcgrl_env_row_layout")
            self._row_layout_cache = lay
        return self._row_layout_cache

    @property
    def env_row_bytes(self) -> int:
        """Bytes of one packed env row (save_envs / load_envs / fork_envs), a multiple of 16."""
        return int(self._row_layout().row_bytes)

    def row_fields(self, rows):
        """Typed views into a [M, env_row_bytes] uint8 tensor of packed rows, one per section this env's rows have:
        grids i8 [M, row_stride], static_mask u8 [M, row_stride], cache u8 [M, cache_stride], records u8
        [M, record_stride], targets f64 [M, K, 2], stats i32 [M, K], holes i32 [M, hole_ints], agent_pos i32
        [M, n_agents, 3], n_step / iteration / changes i32 [M], reward f32 [M], done / changed u8 [M].  Offsets come
        from the library (pcgrl_env_row_layout), so an archive can read or filter saved states, by stats say, without
        loading them."""
        lay = self._row_layout()
        if not torch.is_tensor(rows) or rows.dtype != torch.uint8 or rows.dim() != 2 or rows.shape[1] != lay.row_bytes \
                or rows.stride(1) != 1:
            raise ValueError(f"rows must be a uint8 [M, {lay.row_bytes}] tensor with contiguous rows")
        inner = {"grids": (self.row_stride,), "static_mask": (self.row_stride,), "cache": (self.cache_stride,),
                 "records": (self.record_stride,), "targets": (self.K, 2), "stats": (self.K,),
                 "holes": (self.hole_ints,), "agent_pos": (lay.n_pos, 3)}
        m, out = rows.shape[0], {}
        for name, field, dt in self._ROW_FIELDS:
            off = getattr(lay, field)
            if off < 0:
                continue
            shape = inner.get(name, ())
            nbytes = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
            v = rows[:, off:off + nbytes].view(dt)
            out[name] = v.view(m, *shape) if shape else v[:, 0]
        return out

    def save_envs(self, env_ids=None) -> torch.Tensor:
        """The whole state of envs env_ids (default all) as a new device uint8 tensor [M, env_row_bytes], row j = env
        env_ids[j]: grid, frozen mask, search cache, packed record, per-env targets, stats, holes, every agent's position,
        n_step / iteration / changes and the last reward / done / changed (pcgrl_save_envs).  Indices may repeat and come
        in any order; a bad index raises IndexError before anything is launched (a device tensor costs one reduction and
        one sync).  Not in a row: shared targets, the reset RNG position (seed, epoch) and smb's playthrough-length
        history, which only picks a job class of its solver, never a result."""
        self._check_fresh("save_envs")
        idx = None if env_ids is None else self._check_env_ids(env_ids)
        m = self.n_envs if idx is None else idx.numel()
        rows = torch.empty((m, self.env_row_bytes), dtype=torch.uint8, device=self.device)
        self._save_rows(idx, m, rows)
        self._synced_steps = None
        return rows

    def load_envs(self, rows: torch.Tensor, env_ids=None):
        """Env env_ids[j] (default j) becomes bit for bit the env row j of `rows` was saved from (pcgrl_load_envs); every
        other env is untouched and nothing is reset, auto_reset or not.  rows: a contiguous uint8 [M, env_row_bytes]
        tensor on this env's device, saved by any env with the same row layout (another n_envs, env_offset, seed or
        device after .to(env.device) included).  env_ids: M DISTINCT indices.  A bad or repeated index (IndexError /
        ValueError) or a row saved under another layout (ValueError) raises before anything is launched; each check of
        device data costs one reduction and one sync."""
        self._check_fresh("load_envs")
        lay = self._row_layout()
        if not torch.is_tensor(rows) or rows.dtype != torch.uint8 or rows.dim() != 2 or \
                rows.shape[1] != lay.row_bytes or not rows.is_contiguous() or rows.device != self.device:
            raise ValueError(f"rows must be a contiguous uint8 [M, {lay.row_bytes}] tensor on {self.device}")
        m = rows.shape[0]
        idx = None
        if env_ids is None:
            if m > self.n_envs:
                raise ValueError(f"{m} rows for {self.n_envs} envs")
        else:
            idx = self._check_env_ids(env_ids, distinct=True)
            if idx.numel() != m:
                raise ValueError(f"{m} rows for {idx.numel()} env_ids")
        if m:
            sig = lay.signature - (1 << 32) if lay.signature >= 1 << 31 else lay.signature   # as int32
            want = torch.tensor([sig, lay.row_bytes], dtype=torch.int32, device=self.device)
            if bool((rows[:, :8].view(torch.int32) != want).any()):
                raise ValueError("rows were not saved from an env with this env's row layout (header mismatch)")
            self._load_rows(rows, idx, m)
        self._synced_steps = None

    def fork_envs(self, src_ids, dst_ids):
        """Env dst_ids[j] becomes a copy of env src_ids[j] as it was before the call (save into a reusable buffer, then
        load: two launches).  dst_ids are distinct, src_ids may repeat, and the two may overlap: a beam step overwrites
        the whole shard with copies of its best children.  Bad or repeated indices raise IndexError / ValueError before
        anything is launched.  Nothing is reset."""
        self._check_fresh("fork_envs")
        src = self._check_env_ids(src_ids)
        dst = self._check_env_ids(dst_ids, distinct=True)
        m = dst.numel()
        if src.numel() != m:
            raise ValueError(f"{src.numel()} src_ids for {m} dst_ids")
        if m:
            S = self.env_row_bytes
            if self._fork_buf is None or self._fork_buf.numel() < m * S:
                self._fork_buf = None
                self._fork_buf = torch.empty(m * S, dtype=torch.uint8, device=self.device)
            buf = self._fork_buf[:m * S].view(m, S)
            self._save_rows(src, m, buf)
            self._load_rows(buf, dst, m)     # the library's own rows: no header check
        self._synced_steps = None

    def _save_rows(self, idx, m, rows):
        if m:
            with self._on_device():
                _lib.check(self.lib.pcgrl_save_envs(self._cc, self._st, self.agent_pos.shape[0], _ptr(idx), m,
                                                    rows.data_ptr(), self._stream()), "pcgrl_save_envs")

    def _load_rows(self, rows, idx, m):
        with self._on_device():
            _lib.check(self.lib.pcgrl_load_envs(self._cc, self._st, self.agent_pos.shape[0], rows.data_ptr(), _ptr(idx), m,
                                                self._stream()), "pcgrl_load_envs")

    # ------------------------------------------------------------------ level distances
    def novelty(self, archive_rows: torch.Tensor, k: int, env_ids=None) -> torch.Tensor:
        """Novelty of envs env_ids (default all) against an archive of saved rows (save_envs of an env with this row
        layout): the mean Hamming distance of each env's grid to its k nearest archive grids (level_knn), float32 [M].
        With fewer than k archive rows the mean is over those there are (NaN for an empty archive).  A bad index raises
        IndexError before anything is launched (a device tensor costs one reduction and one sync)."""
        arch = self.row_fields(archive_rows)["grids"]
        queries = self.grids if env_ids is None else self.grids[self._check_env_ids(env_ids).long()]
        dist, _ = level_knn(queries, arch, k=k, cfg=self)
        valid = dist >= 0
        return (dist.clamp(min=0).sum(1).double() / valid.sum(1)).float()

    def diversity(self, group_size: int) -> torch.Tensor:
        """Mean pairwise Hamming distance within each group of group_size consecutive envs (level_diversity of the
        env's own grids), float64 [n_envs / group_size]."""
        return level_diversity(self.grids, group_size, cfg=self)

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

    def _action_layout(self, n=None):
        """(shape, numpy dtype, torch dtype) of one action batch (n rows, default n_envs) for this env's action_kind."""
        N = self.n_envs if n is None else n
        scalar = {4: (np.int32, torch.int32), 1: (np.uint8, torch.uint8), 2: (np.uint16, torch.uint16)}[self._act_elem]
        return {"int32": ((N,), *scalar), "wide_flat": ((N,), *scalar),
                "wide_coords": ((N, self.ndim + 1), np.int32, torch.int32),
                "ca_tiles": ((N, self.row_stride), np.int8, torch.int8),
                "ca_logits": ((N, self.n_tiles * self.cells), np.float32, torch.float32),
                "patch": ((N, int(np.prod(self.act_window or (1,)))), np.int32, torch.int32)}[self.action_kind]

    def _check_actions(self, actions, n=None):
        if not torch.is_tensor(actions) or actions.device != self.device:
            raise TypeError("actions must be a tensor on the env's device (use step_host for host arrays)")
        shape, _, tdt = self._action_layout(n)
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

    def _agent_occupancy(self, agent, dims, dtype, rows=None, acting_pos=None):
        """[N, *dims] (rows: [M] env indices -> [M, *dims]): 1 where any agent stands, in agent `agent`'s window
        (Cropped pads this key with 0).  acting_pos: [M, 3] positions that replace agent `agent`'s own (a lookahead's
        after-state)."""
        nd, dev = self.ndim, self.device
        sel = slice(None) if rows is None else rows.long()
        pos = self.agent_pos[:, sel, :nd].long()
        if acting_pos is not None:
            pos[agent] = acting_pos[:, :nd].long()
        occ = torch.zeros((pos.shape[1], *dims), dtype=dtype, device=dev)
        center = pos[agent]
        half = torch.tensor([d // 2 for d in dims], device=dev)
        lim = torch.tensor(list(dims), device=dev)
        env_idx = torch.arange(pos.shape[1], device=dev)
        for b in range(self.n_agents):
            rel = pos[b] - center + half
            ok = ((rel >= 0) & (rel < lim)).all(dim=1)
            occ[(env_idx[ok],) + tuple(rel[ok, i] for i in range(nd))] = 1
        return occ

    def observe(self, out: torch.Tensor | None = None, dtype=torch.float32, onehot: bool = True, agent: int = 0,
                env_ids=None):
        """The wrapped observation of every env: [N, *obs_dims, channels] (channels last), exactly what
        CroppedImagePCGRLWrapper / ActionMapImagePCGRLWrapper + ControlWrapper return per env.
        dtype: uint8 (no control planes), float32, float64, or float16 / bfloat16 for a policy that runs in half
        precision -- byte for byte the float32 observation converted (round to nearest even), written directly at 2
        bytes per element.  Any other dtype raises TypeError before anything is allocated or launched.
        onehot=False (uint8 only, no controls): the tile codes of the crop instead of their one-hot records --
        Cropped's own output (wrappers.py:407-437: 0 = out of bounds, tile t -> t + 1), one channel, for policies
        that embed the tile themselves (SURVEY 8f rank 3).
        agent: with n_agents > 1, whose crop (every agent sees the shared map around its own position).
        env_ids: a 1-D integer array / tensor of M env indices (any order, duplicates allowed): returns [M, ...],
        row j being row env_ids[j] of the full observation (pcgrl_observe_envs); `out` must then be [M, ...].  An index
        outside [0, N) raises IndexError before anything is launched (a device tensor costs one reduction and one
        sync for that check)."""
        rows = None if env_ids is None else self._check_env_ids(env_ids)
        return self._observe(out, dtype, onehot, agent, rows)

    def _check_env_ids(self, env_ids, distinct=False):
        """-> int32 device tensor of validated env indices (distinct: a repeated index raises ValueError)."""
        if torch.is_tensor(env_ids):
            t = env_ids
            if t.dim() != 1 or (t.numel() and (t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool)):
                raise IndexError(f"env_ids must be a 1-D integer index, got {tuple(t.shape)} {t.dtype}")
            if t.numel():
                if distinct:    # one sort gives the range and the repeats, read back in one sync
                    srt = t.to(torch.int64).sort().values
                    lo, hi, rep = torch.stack([srt[0], srt[-1], (srt[1:] == srt[:-1]).any().to(torch.int64)]).tolist()
                else:
                    lo, hi = torch.stack(torch.aminmax(t)).tolist()      # host tensors: no device work
                    rep = 0
                if lo < 0 or hi >= self.n_envs:
                    raise IndexError(f"env_ids in [{lo}, {hi}] outside [0, {self.n_envs})")
                if rep:
                    raise ValueError("env_ids repeat an env index")
            return t.to(device=self.device, dtype=torch.int32).contiguous()
        a = np.asarray(env_ids)
        if a.ndim != 1 or (a.size and a.dtype.kind not in "iu"):
            raise IndexError(f"env_ids must be a 1-D integer index, got shape {a.shape} {a.dtype}")
        if a.size and (int(a.min()) < 0 or int(a.max()) >= self.n_envs):
            raise IndexError(f"env_ids in [{int(a.min())}, {int(a.max())}] outside [0, {self.n_envs})")
        if distinct and np.unique(a).size != a.size:
            raise ValueError("env_ids repeat an env index")
        return torch.from_numpy(a.astype(np.int32)).to(self.device)

    def _observe_envs(self, rows, out=None, dtype=torch.float32, onehot: bool = True, agent: int = 0):
        """observe(env_ids=rows) without the range check, for indices this library produced itself (a nonzero of the
        done flags, an env the caller just reset)."""
        return self._observe(out, dtype, onehot, agent, rows.to(device=self.device, dtype=torch.int32).contiguous())

    def _observe(self, out, dtype, onehot, agent, rows):
        final, out, oa = self._obs_buffers(self.n_envs if rows is None else rows.numel(), out, dtype, onehot)
        st = self._agent_state(agent)
        if rows is None:
            with self._on_device():
                _lib.check(self.lib.pcgrl_observe(self._cc, st, oa, self._stream()), "pcgrl_observe")
        elif rows.numel():
            with self._on_device():
                _lib.check(self.lib.pcgrl_observe_envs(self._cc, st, oa, rows.data_ptr(), rows.numel(), self._stream()),
                           "pcgrl_observe_envs")
        occ = self._agent_occupancy(agent, out.shape[1:-1], out.dtype, rows) if self.show_agents else None
        return self._obs_finish(final, out, occ)

    def _obs_buffers(self, m, out, dtype, onehot):
        """Checks and buffers of an observation of m rows, before anything is launched: -> (final, out, oa).  The
        kernel writes `out` (every channel but the occupancy plane) as pcgrl_obs_args `oa` describes; `final` is the
        caller's tensor that _obs_finish completes, or None."""
        if self.ctrl_metrics:
            self._check_fresh("observe with control planes")
        if not onehot:
            if self.ctrl_metrics or (out is not None and out.dtype != torch.uint8):
                raise ValueError("onehot=False is a uint8 observation without control planes")
            dtype = torch.uint8
        shape = (m, *self.obs_shape(onehot))
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
        self._check_obs_dtype(dtype if out is None else out.dtype)
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
        oa.out_kind = self.OBS_KINDS[out.dtype] if onehot else 3
        oa.out = out.data_ptr()
        oa.static_channel = 1 if self.static_mask is not None else 0
        return final, out, oa

    # element type of a one-hot observation -> pcgrl_obs_args.out_kind (tile codes are uint8, kind 3).  float16 and
    # bfloat16 are the float32 observation rounded to nearest even, for policies that run in half precision.
    OBS_KINDS = {torch.uint8: 0, torch.float32: 1, torch.float64: 2, torch.float16: 5, torch.bfloat16: 6}

    def _check_obs_dtype(self, dtype):
        if dtype not in self.OBS_KINDS:
            raise TypeError(f"observation dtype {dtype} is not one of {', '.join(map(str, self.OBS_KINDS))}")

    def _obs_finish(self, final, out, occ):
        """The observation: `out` with the occupancy plane `occ` appended (show_agents), into `final` if given."""
        if not self.show_agents:
            return out
        if final is None:
            return torch.cat([out, occ[..., None]], dim=-1)
        final[..., :-1] = out
        final[..., -1] = occ
        return final

    STATUS_BITS = (
        (1, ValueError, "an action outside the action space reached pcgrl_step (ignored on device)"),
        (2, IndexError, "minecraft_3D_maze: the reference raises IndexError on this map (helper_3D.py:531: a recorded "
                        "x or y >= depth); the stats of that env are not meaningful"),
        (4, RuntimeError, "a search workspace overflowed: the stats of at least one env are NOT the reference's "
                          "(parity lost) -- report the map"),
        (8, RuntimeError, "sokoban: a level with more than 15 crates met the solver preconditions; a packed solver "
                          "state holds 15, so its dist-win / sol-length were not computed"),
        (16, OverflowError, "a stat did not fit the packed result record (record_stat_bytes too small)"),
        (64, IndexError, "observe: env index out of range (pcgrl_observe_envs loaded nothing through it)"),
        (128, IndexError, "lookahead: env index out of range (pcgrl_lookahead loaded nothing through it)"),
        (256, IndexError, "step: env index out of range (pcgrl_step_envs loaded and wrote nothing through it)"),
        (512, IndexError, "save / load / fork: env index out of range (pcgrl_save_envs wrote a zero row for it, "
                          "pcgrl_load_envs wrote nothing)"),
        (1024, ValueError, "load: a row's header does not match this env's row layout (nothing of it was loaded)"),
    )

    def check_status(self):
        """Raise the error that matches the device status word (include/pcgrl_b200.h, pcgrl_state.status); one D2H
        sync.  Parity-relevant conditions (workspace overflow, crate limit) outrank a bad action."""
        s = int(self.status.item())
        if not s:
            return
        self.status.zero_()
        for bit, exc, msg in sorted(self.STATUS_BITS, key=lambda b: b[0] not in (4, 8)):
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


# ---------------------------------------------------------------------- level distances (pcgrl_level_*)
def _level_config(cfg):
    """The pcgrl_config whose dims and n_tiles give the level geometry: an env's own, or one built from a config."""
    if isinstance(cfg, BatchedPcgrlEnv):
        return cfg._cc
    c = normalise(cfg)
    spec = get_spec(c.problem, c.map_shape)
    cc = _lib.Config()
    cc.abi_version = _lib.PCGRL_ABI_VERSION
    cc.problem = _lib.PROB_IDS[c.problem]
    cc.representation = _lib.REP_IDS["narrow"]
    cc.action_kind = _lib.ACT_INT32
    cc.ndim = len(c.map_shape)
    for i in range(3):
        cc.dims[i] = c.map_shape[i] if i < cc.ndim else 1
    cc.n_tiles, cc.n_stats = spec.n_tiles, len(spec.stat_names)
    cc.max_iterations, cc.max_changes = 1, -1
    _lib.check(_lib.load().pcgrl_config_check(cc), "pcgrl_config_check")
    return cc


def _levels(t, cc, env, what):
    """-> (levels tensor, byte stride) of [M, >= cells] int8 / uint8 grids (env grids, [M, cells] maps, a row_fields
    'grids' view), or of an env's saved rows [M, env_row_bytes] when cfg is that env."""
    cells = int(np.prod([cc.dims[i] for i in range(cc.ndim)]))
    if not torch.is_tensor(t) or t.dtype not in (torch.int8, torch.uint8) or t.dim() != 2:
        raise ValueError(f"{what} must be a 2-D int8 / uint8 tensor of levels")
    if env is not None and t.dtype == torch.uint8 and t.shape[1] == env.env_row_bytes:
        t = env.row_fields(t)["grids"]
    if not t.is_cuda:
        raise ValueError(f"{what} must be on a CUDA device")
    stride = t.stride(0) if t.shape[0] > 1 else cells
    if t.shape[1] < cells or (t.shape[1] > 1 and t.stride(1) != 1) or stride < cells:
        raise ValueError(f"{what} must hold one level of {cells} tile codes per row, with contiguous rows")
    return t, stride


def _level_call(a, b, cfg):
    cc = _level_config(cfg)
    env = cfg if isinstance(cfg, BatchedPcgrlEnv) else None
    a, sa = _levels(a, cc, env, "a")
    b, sb = (a, sa) if b is None else _levels(b, cc, env, "b")
    if a.device != b.device:
        raise ValueError(f"a is on {a.device}, b on {b.device}")
    return cc, a, sa, b, sb


def level_distances(a: torch.Tensor, b: torch.Tensor | None = None, *, cfg) -> torch.Tensor:
    """Hamming distances between levels: int32 [M, N], out[i, j] = the number of cells where level a[i] and level b[j]
    (default: a) hold different tile codes.  a, b: [M, cells] or [M, row_stride] int8 / uint8 grids (only the first cells
    bytes of a row count), a row_fields(rows)['grids'] view, or, when cfg is a BatchedPcgrlEnv, saved rows of it.  cfg:
    a make_config config or an env; it gives the map shape and tile count.  Meant for small problems: the output is
    M * N * 4 bytes; level_knn never writes it."""
    cc, a, sa, b, sb = _level_call(a, b, cfg)
    lib, m, n = _lib.load(), a.shape[0], b.shape[0]
    out = torch.empty((m, n), dtype=torch.int32, device=a.device)
    work = torch.empty(max(int(lib.pcgrl_level_work_bytes(cc, m, n, 0)), 16), dtype=torch.uint8, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(lib.pcgrl_level_distances(cc, a.data_ptr(), m, sa, b.data_ptr(), n, sb, out.data_ptr(),
                                             work.data_ptr(), torch.cuda.current_stream().cuda_stream),
                   "pcgrl_level_distances")
    return out


def level_knn(a: torch.Tensor, b: torch.Tensor | None = None, *, k: int, cfg, exclude_self: bool = False,
              self_offset: int = 0):
    """The k nearest levels of b (default: a) to every level of a, 1 <= k <= 64: (dist, idx) int32 [M, k], each row in
    ascending distance and, on equal distance, ascending index of b, so the result is deterministic.  exclude_self:
    query i never picks level i + self_offset of b (novelty within a population: b None, offset 0).  With fewer than k
    candidates a row ends in -1 / -1.  Inputs as for level_distances; no M x N matrix is formed."""
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= k <= 64:
        raise ValueError(f"k must be an integer in [1, 64], got {k!r}")
    if exclude_self and self_offset < 0:
        raise ValueError("self_offset must be >= 0")
    cc, a, sa, b, sb = _level_call(a, b, cfg)
    lib, m, n = _lib.load(), a.shape[0], b.shape[0]
    dist = torch.empty((m, k), dtype=torch.int32, device=a.device)
    idx = torch.empty((m, k), dtype=torch.int32, device=a.device)
    work = torch.empty(max(int(lib.pcgrl_level_work_bytes(cc, m, n, k)), 16), dtype=torch.uint8, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(lib.pcgrl_level_knn(cc, a.data_ptr(), m, sa, b.data_ptr(), n, sb, int(k),
                                       int(self_offset) if exclude_self else -1, dist.data_ptr(), idx.data_ptr(),
                                       work.data_ptr(), torch.cuda.current_stream().cuda_stream), "pcgrl_level_knn")
    return dist, idx


def level_diversity(a: torch.Tensor, group_size: int, *, cfg) -> torch.Tensor:
    """Diversity of consecutive groups of group_size levels (group_size >= 2 divides M): float64 [M / group_size], the
    mean Hamming distance over the unordered pairs of each group (the int64 pair sum from the device over
    S (S - 1) / 2).  Inputs as for level_distances."""
    cc, a, sa, _, _ = _level_call(a, None, cfg)
    lib, m, s = _lib.load(), a.shape[0], int(group_size)
    if s < 2 or m % s:
        raise ValueError(f"group_size {group_size} must be >= 2 and divide {m}")
    sums = torch.empty(m // s, dtype=torch.int64, device=a.device)
    work = torch.empty(max(int(lib.pcgrl_level_work_bytes(cc, m, 0, 0)), 16), dtype=torch.uint8, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(lib.pcgrl_level_group_diversity(cc, a.data_ptr(), m, sa, s, sums.data_ptr(), work.data_ptr(),
                                                   torch.cuda.current_stream().cuda_stream),
                   "pcgrl_level_group_diversity")
    return sums.double() / (s * (s - 1) // 2)
