"""PcgrlVectorEnv: the batched seam for RL trainers (SURVEY.md 8b / 8f-3).

A gymnasium.vector-style API over BatchedPcgrlEnv: one object owns N GPU envs, `step(actions)` returns
batched tensors that stay on the device (the policy runs there too), with auto-reset.  It replaces the
reference's N Python envs per Ray rollout worker (rl/utils.py:402-415) with one launch per step.
"""
from __future__ import annotations

import numpy as np
import torch

from . import spaces
from .batched_env import BatchedPcgrlEnv


class PcgrlVectorEnv:
    """shards > 1: the N envs live in `shards` independent BatchedPcgrlEnv objects (consecutive env ranges, the same
    maps as one shard would draw: resets are counter-based on the global env index), each stepped and observed on
    its own CUDA stream.  The binary step is bound by the integer pipes and the observation writer by HBM, so one
    shard's search runs beside another shard's observation writes instead of the two taking turns
    (scripts/bench_rl_loop.py).  Outputs are the same [N, ...] tensors either way."""

    def __init__(self, cfg, num_envs: int, device="cuda:0", obs_dtype=torch.float32, env_offset=0, seed=0,
                 uniform_targets: bool | None = None, shards: int = 1, onehot: bool = True):
        shards = max(1, min(int(shards), num_envs))
        per = -(-num_envs // shards)
        self._ranges = [(lo, min(num_envs, lo + per)) for lo in range(0, num_envs, per)]
        self.shards = [BatchedPcgrlEnv(cfg, hi - lo, device=device, env_offset=env_offset + lo, seed=seed, auto_reset=False)
                       for lo, hi in self._ranges]
        self.env = self.shards[0]          # metadata (spaces, names, bounds); the only shard when shards == 1
        self.num_envs = num_envs
        # onehot=False: observations are the crop's tile codes, one uint8 per pixel (Cropped's own output, a third of
        # the one-hot bytes); control_pcgrl_b200.policy_input.conv_input_from_codes expands them inside the policy
        self.onehot = bool(onehot)
        if not self.onehot:
            obs_dtype = torch.uint8
        self.obs_dtype = obs_dtype
        b = self.env
        if b.ctrl_metrics and obs_dtype == torch.uint8:
            raise ValueError("target channels are fractional: use a float obs_dtype with controls")
        self.uniform_targets = bool(b.ctrl_metrics) if uniform_targets is None else uniform_targets
        shp = b.obs_shape(self.onehot)
        self.single_observation_space = spaces.Box(0, 1 if self.onehot else b.n_tiles + 1, shape=shp, dtype=np.float32)
        rep = b.representation
        if rep == "narrow":
            self.single_action_space = spaces.Discrete(b.n_tiles)
        elif rep == "turtle":
            self.single_action_space = spaces.Discrete(4 + b.n_tiles)
        elif rep == "wide":
            self.single_action_space = spaces.Discrete(b.obs_window[0] * b.obs_window[1] * b.n_tiles)
        else:
            self.single_action_space = spaces.Box(0, 1, shape=(b.n_tiles * b.cells,), dtype=np.float32)
        self._obs = torch.empty((num_envs, *shp), dtype=obs_dtype, device=b.device)
        self.episode_return = torch.zeros(num_envs, dtype=torch.float64, device=b.device)
        self.episode_length = torch.zeros(num_envs, dtype=torch.int32, device=b.device)
        if len(self.shards) > 1:
            self._streams = [torch.cuda.Stream(device=b.device) for _ in self.shards]
            self._reward = torch.zeros(num_envs, dtype=torch.float32, device=b.device)
            self._done = torch.zeros(num_envs, dtype=torch.uint8, device=b.device)

    def _on_shards(self, fn):
        """fn(i, shard, lo, hi) for every shard on its own stream; the caller's stream waits for all of them."""
        cur = torch.cuda.current_stream(self.env.device)
        for i, (b, st, (lo, hi)) in enumerate(zip(self.shards, self._streams, self._ranges)):
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                fn(i, b, lo, hi)
        for st in self._streams:
            cur.wait_stream(st)

    def reset(self, grids=None, pos=None):
        if len(self.shards) == 1:
            if self.uniform_targets:
                self.env.sample_uniform_targets()
            self.env.reset(grids=grids, pos=pos)
            self.episode_return.zero_()
            self.episode_length.zero_()
            return self.env.observe(out=self._obs, onehot=self.onehot), {}

        def one(i, b, lo, hi):
            if self.uniform_targets:
                b.sample_uniform_targets()
            b.reset(grids=None if grids is None else grids[lo:hi], pos=None if pos is None else pos[lo:hi])
            b.observe(out=self._obs[lo:hi], onehot=self.onehot)
        self._on_shards(one)
        self.episode_return.zero_()
        self.episode_length.zero_()
        return self._obs, {}

    def _step_shard(self, b, actions, lo, hi, infos):
        """One shard's step + auto-reset + observation (on the current stream); -> (reward, done) of the shard."""
        reward, done = b.step(actions)
        ret, length = self.episode_return[lo:hi], self.episode_length[lo:hi]
        ret += reward.double()
        length += 1
        # lock-step episodes (no change budget, every env reset together): the episode end is known on the host
        # without a device-to-host sync, and STAYS known afterwards because the reset below is a full one
        lock_step = b.max_changes is None and b._synced_steps is not None
        if lock_step:
            any_done = b._synced_steps > b.max_iterations
        else:
            ended = done.nonzero().squeeze(1)        # the step's one host sync
            any_done = ended.numel() > 0
        if any_done:
            d = done.bool()
            # the terminal observations, before the targets are redrawn and the envs reset: their target / value
            # planes show the targets and stats the episodes ended with
            if lock_step:
                final_obs = b.observe(dtype=self.obs_dtype, onehot=self.onehot)
                final_idx = torch.arange(lo, hi, dtype=torch.int64, device=b.device)
            else:
                final_obs = b._observe_envs(ended, dtype=self.obs_dtype, onehot=self.onehot)
                final_idx = ended + lo
            infos.append((lo, {"final_stats": b.stats.clone(), "final_return": ret.clone(),
                               "final_length": length.clone(), "_final": d,
                               "final_obs": final_obs, "final_idx": final_idx}))
            if lock_step:
                if self.uniform_targets:
                    b.sample_uniform_targets()
                b.reset()
                ret.zero_()
                length.zero_()
            else:
                if self.uniform_targets:
                    keep = b.targets.clone()
                    b.sample_uniform_targets()
                    b.targets[~d] = keep[~d]
                b.reset(mask=done)
                ret[d] = 0
                length[d] = 0
        b.observe(out=self._obs[lo:hi], onehot=self.onehot)
        return reward, done

    def step(self, actions: torch.Tensor):
        """-> obs, reward, terminated(False), truncated(done), info; finished envs are reset in place and
        their `obs` row is the first observation of the new episode (gymnasium autoreset semantics);
        info carries the final stats of finished episodes (rows where info["_final"] is set; with shards > 1 the
        rows of ranges that saw no episode end are zero), and their terminal observations as compact rows:
        info["final_obs"] [M, *obs_shape] is the observation of env info["final_idx"][j] ([M] int64, ascending) after
        its last step, before its reset -- what a value bootstrap of the truncated episode needs.  reward / done are
        the env's own output tensors: a reset leaves them alone (include/pcgrl_b200.h, pcgrl_reset), so they need no
        copies."""
        infos = []
        if len(self.shards) == 1:
            reward, done = self._step_shard(self.env, actions, 0, self.num_envs, infos)
            return self._obs, reward, torch.zeros_like(done), done, (infos[0][1] if infos else {})

        def one(i, b, lo, hi):
            r, d = self._step_shard(b, actions[lo:hi], lo, hi, infos)
            self._reward[lo:hi].copy_(r)
            self._done[lo:hi].copy_(d)
        self._on_shards(one)
        info = {}
        if infos:      # some shard saw an episode end: whole-batch tensors, rows of the other shards not final
            K = self.env.K
            info = {"final_stats": torch.zeros((self.num_envs, K), dtype=torch.int32, device=self.env.device),
                    "final_return": torch.zeros(self.num_envs, dtype=torch.float64, device=self.env.device),
                    "final_length": torch.zeros(self.num_envs, dtype=torch.int32, device=self.env.device),
                    "_final": torch.zeros(self.num_envs, dtype=torch.bool, device=self.env.device)}
            for lo, part in infos:
                for k, v in part.items():
                    if k not in ("final_obs", "final_idx"):
                        info[k][lo:lo + v.shape[0]] = v
            # the ranges' compact rows in range order: final_idx stays ascending
            info["final_obs"] = torch.cat([part["final_obs"] for _, part in infos])
            info["final_idx"] = torch.cat([part["final_idx"] for _, part in infos])
        return self._obs, self._reward, torch.zeros_like(self._done), self._done, info


# ------------------------------------------------------------------------------------------------------------------
# RLlib seam (SURVEY.md 8b / 8f rank 3): rl/train.py:251 registers `make_env` and RLlib then builds
# num_rollout_workers x num_envs_per_worker Python envs (rl/utils.py:402-415), wrapping each worker's list in its own
# _VectorizedGymEnv.  This class is that VectorEnv directly: one object, N grids on the GPU, the same
# vector_reset / reset_at / restart_at / vector_step / get_sub_environments surface, host (numpy) observations.
# ------------------------------------------------------------------------------------------------------------------
class _SubEnvView:
    """What the reference's callbacks and evaluation code read from a sub-environment (rl/callbacks.py:30-116,
    rl/evaluate.py): metrics, targets and bounds of env `index` of the batch."""

    def __init__(self, owner, index):
        self._o, self._i = owner, index

    @property
    def unwrapped(self):
        return self

    @property
    def metrics(self):
        return self._o.env.stats_dict(self._i)

    _rep_stats = metrics

    @property
    def ctrl_metrics(self):
        return self._o.env.ctrl_metrics

    @property
    def cond_bounds(self):
        return self._o.env.cond_bounds

    @property
    def static_trgs(self):
        return self._o.env.static_trgs

    @property
    def metric_trgs(self):
        b = self._o.env
        row = b.targets[self._i if b.ctrl_metrics else 0].cpu().numpy()
        return {k: (float(row[j, 0]) if np.isnan(row[j, 1]) else (float(row[j, 0]), float(row[j, 1])))
                for j, k in enumerate(b.stat_names) if k in b.all_metrics}

    def get_map(self):
        return self._o.env.maps[self._i].cpu().numpy()


def _rllib_base():
    try:                                             # a real ray install (absent from this image)
        from ray.rllib.env.vector_env import VectorEnv
        return VectorEnv
    except Exception:                                # noqa: BLE001 -- same surface without the base class
        return object


def make_rllib_vector_env(cfg, num_envs: int, device="cuda:0", obs_dtype=np.float32, seed=0, env_offset=0):
    """-> an RLlib `VectorEnv` (a subclass of ray.rllib.env.vector_env.VectorEnv when ray is importable) whose
    `num_envs` sub-environments are one BatchedPcgrlEnv shard.  Register it instead of the per-env creator:

        register_env("pcgrl", lambda env_ctx: make_rllib_vector_env(env_ctx, env_ctx["num_envs_per_worker"]))

    Observations are what make_env's wrapper stack returns per env (rl/envs.py:28-66: cropped / full one-hot image
    with the ControlWrapper target planes), as numpy rows of one pinned host array of obs_dtype (uint8, float32,
    float64, or float16: half the bytes of float32 over PCIe; numpy has no bfloat16); rewards / truncation flags /
    info stats come back in one packed record array (compact host I/O)."""
    Base = _rllib_base()

    class PcgrlRLlibVectorEnv(Base):
        def __init__(self):
            self.env = BatchedPcgrlEnv(cfg, num_envs, device=device, env_offset=env_offset, seed=seed,
                                       auto_reset=False, compact_host_io=True)
            b = self.env
            shp = b.obs_shape()
            tdt = {np.float32: torch.float32, np.float64: torch.float64, np.float16: torch.float16,
                   np.uint8: torch.uint8}[np.dtype(obs_dtype).type]
            self.observation_space = spaces.Box(0, 1, shape=shp, dtype=obs_dtype)
            rep = b.representation
            if b.act_window is not None:
                self.action_space = spaces.MultiDiscrete([b.n_tiles] * int(np.prod(b.act_window)))
            elif rep == "narrow":
                self.action_space = spaces.Discrete(b.n_tiles)
            elif rep == "turtle":
                self.action_space = spaces.Discrete(4 + b.n_tiles)
            elif rep == "wide":
                self.action_space = spaces.Discrete(b.obs_window[0] * b.obs_window[1] * b.n_tiles)
            else:
                self.action_space = spaces.Box(0, 1, shape=(b.n_tiles * b.cells,), dtype=np.float32)
            if Base is not object:
                super().__init__(self.observation_space, self.action_space, num_envs)
            self.num_envs = num_envs
            self._obs_dev = torch.empty((num_envs, *shp), dtype=tdt, device=b.device)
            self._obs_host = torch.empty((num_envs, *shp), dtype=tdt, pin_memory=True)      # current observations
            # first observations after the auto-reset of vector_step, compact: row _new_row[i] for env i
            self._new_host = torch.empty((num_envs, *shp), dtype=tdt, pin_memory=True)
            self._new_row = np.zeros(num_envs, dtype=np.int64)
            self._fresh = np.zeros(num_envs, dtype=bool)    # envs reset inside the last vector_step, not yet handed out
            self._views = [_SubEnvView(self, i) for i in range(num_envs)]

        def _observe_into(self, host):
            self.env.observe(out=self._obs_dev)
            host.copy_(self._obs_dev, non_blocking=True)
            torch.cuda.current_stream(self.env.device).synchronize()
            return host.numpy()

        def _observe_rows_into(self, ids, host):
            """Observe the envs `ids` only (numpy int array) into host[:len(ids)]: M rows written, M rows copied."""
            m = len(ids)
            rows = torch.from_numpy(np.ascontiguousarray(ids, dtype=np.int32)).to(self.env.device)
            self.env._observe_envs(rows, out=self._obs_dev[:m])
            host[:m].copy_(self._obs_dev[:m], non_blocking=True)
            torch.cuda.current_stream(self.env.device).synchronize()

        def vector_reset(self, *, seeds=None, options=None):
            b = self.env
            if seeds is not None and seeds[0] is not None:
                b.seed = int(seeds[0])
            if b.ctrl_metrics:
                b.sample_uniform_targets()
            b.reset()
            self._fresh[:] = False
            obs = self._observe_into(self._obs_host)
            return [obs[i] for i in range(self.num_envs)], [{} for _ in range(self.num_envs)]

        def reset_at(self, index=None, *, seed=None, options=None):
            i = 0 if index is None else int(index)
            if self._fresh[i]:                     # already reset (with every other finished env) by vector_step
                self._fresh[i] = False
                self._obs_host[i].copy_(self._new_host[self._new_row[i]])
                return self._obs_host.numpy()[i], {}
            mask = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.env.device)
            mask[i] = 1
            self.env.reset(mask=mask)
            self._observe_rows_into(np.array([i]), self._obs_host[i:i + 1])
            return self._obs_host.numpy()[i], {}

        def restart_at(self, index=None):
            self.reset_at(index)

        def vector_step(self, actions):
            b = self.env
            shape, dt, _ = b._action_layout()
            r, d, s = b.step_host(np.asarray(actions).astype(dt, copy=False).reshape(shape))
            obs = self._observe_into(self._obs_host)
            rewards, dones = r.tolist(), d.astype(bool).tolist()
            names = b.stat_names
            it = b.iteration.cpu().numpy()
            infos = [dict(zip(names, row), iterations=int(k), max_iterations=b.max_iterations)
                     for row, k in zip(s.tolist(), it.tolist())]
            if d.any():
                # RLlib calls reset_at(i) for every finished env next: reset them all in ONE launch now and keep
                # their first observations ready (the terminal observations above are already on the host)
                self._fresh[:] = d.astype(bool)
                ids = np.flatnonzero(self._fresh)
                self._new_row[ids] = np.arange(len(ids))
                b.reset(mask=b.done)
                self._observe_rows_into(ids, self._new_host)
            return [obs[i] for i in range(self.num_envs)], rewards, [False] * self.num_envs, dones, infos

        def get_sub_environments(self):
            return self._views

        def try_render_at(self, index=None):
            return None

    return PcgrlRLlibVectorEnv()
