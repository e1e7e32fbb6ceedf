"""GPU: the terminal observations PcgrlVectorEnv hands out (info["final_obs"] / info["final_idx"]) and the row-wise
observations of the RLlib seam, against a twin BatchedPcgrlEnv stepped by hand and observed before each reset."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CONFIGS = {   # id -> (problem, rep, make_config kwargs, PcgrlVectorEnv kwargs)
    "binary_narrow_lockstep": ("binary", "narrow", dict(max_board_scans=0.05), dict(obs_dtype=torch.uint8)),
    # a change budget of 12 edits against 51 iterations: episodes end on many different steps
    "binary_narrow_changes": ("binary", "narrow", dict(max_board_scans=0.2, change_percentage=0.05),
                              dict(obs_dtype=torch.float32)),
    "zelda_turtle_changes": ("zelda", "turtle", dict(max_board_scans=0.1, change_percentage=0.3),
                             dict(obs_dtype=torch.uint8)),
    "binary_wide_controls": ("binary", "wide", dict(max_board_scans=0.03, controls=["regions", "path-length"]),
                             dict(obs_dtype=torch.float32, uniform_targets=True)),
    "binary_narrow_controls_changes": ("binary", "narrow", dict(max_board_scans=0.2, change_percentage=0.05,
                                                                controls=["path-length"]),
                                       dict(obs_dtype=torch.float64, uniform_targets=True)),
    "zelda_codes_changes": ("zelda", "narrow", dict(max_board_scans=0.1, change_percentage=0.3), dict(onehot=False)),
}


def _run(cfg_id, n, shards, steps, seed=5):
    """Steps a PcgrlVectorEnv and a hand-stepped twin with the same actions; checks every final observation against
    the twin's observe() before its reset, and returns what the vector env handed out."""
    import control_pcgrl_b200 as P
    from control_pcgrl_b200.vector_env import PcgrlVectorEnv
    problem, rep, ckw, vkw = CONFIGS[cfg_id]
    cfg = P.make_config(problem, rep, **ckw)
    venv = PcgrlVectorEnv(cfg, n, seed=seed, shards=shards, **vkw)
    twin = P.BatchedPcgrlEnv(cfg, n, seed=seed)
    dtype, onehot = venv.obs_dtype, venv.onehot

    def targets():
        return torch.cat([b.targets for b in venv.shards]) if twin.ctrl_metrics else venv.env.targets

    obs, _ = venv.reset()
    twin.reset()
    twin.targets.copy_(targets())
    assert torch.equal(obs, twin.observe(dtype=dtype, onehot=onehot))
    n_act = venv.single_action_space.n
    gen = torch.Generator(device=obs.device).manual_seed(seed)
    record, ends = [], 0
    for t in range(steps):
        act = torch.randint(0, n_act, (n,), generator=gen, device=obs.device, dtype=torch.int32)
        obs, rew, _, done, info = venv.step(act)
        r2, d2 = twin.step(act)
        assert torch.equal(rew, r2) and torch.equal(done, d2), t
        terminal = twin.observe(dtype=dtype, onehot=onehot)      # before the twin's reset: its episodes' last frame
        if d2.any():
            ends += 1
            fi, fo = info["final_idx"], info["final_obs"]
            assert fi.dtype == torch.int64 and fo.dtype == dtype and tuple(fo.shape) == (fi.numel(), *obs.shape[1:])
            assert torch.equal(fi, d2.nonzero().squeeze(1)), t                # ascending, exactly the finished envs
            assert bool(info["_final"][fi].all())
            assert torch.equal(fo, terminal[fi]), t
            record.append((t, fi.clone(), fo.clone()))
            if twin.max_changes is None and twin._synced_steps is not None:
                twin.reset()
            else:
                twin.reset(mask=d2)
            twin.targets.copy_(targets())
        else:
            assert "final_obs" not in info
        assert torch.equal(obs, twin.observe(dtype=dtype, onehot=onehot)), t
    assert ends >= 2
    return record


@pytest.mark.parametrize("cfg_id", list(CONFIGS))
def test_final_obs_equals_twin_before_reset(cfg_id):
    _run(cfg_id, 517, 1, 45)


@pytest.mark.parametrize("cfg_id", ["binary_narrow_lockstep", "zelda_turtle_changes", "zelda_codes_changes"])
def test_final_obs_sharded_equals_one_shard(cfg_id):
    """shards=3: each range observes its own finals on its stream; concatenated in range order they are the one-shard
    rows bit for bit (the sharded run is checked against its own twin as well).  No control configs here: each shard
    draws its own uniform targets, so their target planes differ from the one-shard draw by design."""
    one = _run(cfg_id, 5_003, 1, 30)
    many = _run(cfg_id, 5_003, 3, 30)
    assert len(one) == len(many)
    for (t1, i1, o1), (t2, i2, o2) in zip(one, many):
        assert t1 == t2 and torch.equal(i1, i2) and torch.equal(o1, o2), t1


def test_rllib_seam_observes_only_the_rows_it_hands_out(monkeypatch):
    """vector_step observes the N terminal rows plus the M fresh rows of the envs it reset, and reset_at of a running
    env observes one row; the outputs are the twin's."""
    import control_pcgrl_b200 as P
    from control_pcgrl_b200.batched_env import BatchedPcgrlEnv
    rows_observed = []
    real = BatchedPcgrlEnv._observe

    def spy(self, out, dtype, onehot, agent, rows):
        if self is venv.env:
            rows_observed.append(self.n_envs if rows is None else rows.numel())
        return real(self, out, dtype, onehot, agent, rows)

    n = 64
    cfg = P.make_config("binary", "narrow", max_board_scans=0.05, change_percentage=0.2, controls=["regions"])
    venv = P.make_rllib_vector_env(cfg, n, seed=4, obs_dtype=np.float32)
    twin = P.BatchedPcgrlEnv(cfg, n, seed=4)
    obs, _ = venv.vector_reset()
    twin.targets.copy_(venv.env.targets)
    twin.reset()
    np.testing.assert_array_equal(np.stack(obs), twin.observe().cpu().numpy())
    monkeypatch.setattr(BatchedPcgrlEnv, "_observe", spy)
    rng = np.random.default_rng(0)
    finished = 0
    for t in range(40):
        acts = [int(a) for a in rng.integers(0, 2, size=n)]
        rows_observed.clear()
        obs, rew, _, trunc, _ = venv.vector_step(acts)
        twin.step(torch.tensor(acts, dtype=torch.int32, device=twin.device))
        np.testing.assert_array_equal(np.stack(obs), twin.observe().cpu().numpy())
        m = int(np.sum(trunc))
        assert sum(rows_observed) <= n + m and len(rows_observed) == (2 if m else 1), (t, rows_observed)
        if m:
            twin.reset(mask=twin.done)
            first = twin.observe().cpu().numpy()
            for i in np.flatnonzero(trunc):
                o, _ = venv.reset_at(int(i))
                np.testing.assert_array_equal(o, first[i])
                finished += 1
    assert finished >= n
    # reset_at of a running env: one row observed, the twin's single-env reset
    rows_observed.clear()
    o, _ = venv.reset_at(3)
    assert rows_observed == [1]
    mask = torch.zeros(n, dtype=torch.uint8, device=twin.device)
    mask[3] = 1
    twin.reset(mask=mask)
    np.testing.assert_array_equal(o, twin.observe().cpu().numpy()[3])
