"""Stepping a chosen subset of envs in place (pcgrl_step_envs, BatchedPcgrlEnv.step(env_ids=...)) against a twin env.

For every config of the lookahead suite, after a few random steps and a masked reset (some envs one iteration or one
change from done): env A steps M random distinct envs in random order; twin B, restored from A's state before that
step, takes a full step with the same actions on the listed rows and then gets every unlisted row of every state
tensor back from the snapshot.  A and B must then agree bit for bit on every state tensor and every output, and again
after identical full steps (hidden work-list or scratch state would show there).  Then: long sequences of subset
steps with auto-reset mixed with full steps, lookahead and observe; a large shard; argument validation and the
device-side index guard."""
import numpy as np
import pytest
import torch

import control_pcgrl_b200 as P
from tests.test_gpu_lookahead import CASES, _actions, _make, _prepare

pytestmark = pytest.mark.gpu

# every tensor a step can touch, and the ones it reads
STATE = ("grids", "agent_pos", "n_step", "iteration", "changes", "stats", "targets", "reward", "done", "changed",
         "records", "cache", "static_mask", "holes")


def _snapshot(env):
    return {k: getattr(env, k).clone() for k in STATE if getattr(env, k) is not None}


def _bits(t):
    return t.reshape(-1).view(torch.uint8)     # bytewise: targets hold NaN, rewards are compared bit for bit


def _assert_same(a, b, what):
    for k in STATE:
        x, y = getattr(a, k), getattr(b, k)
        assert (x is None) == (y is None), (what, k)
        if x is not None:
            assert torch.equal(_bits(x), _bits(y)), (what, k)


def _restore_unlisted(env, snap, ids):
    """Every row of every state tensor that is not in ids gets its snapshot value back."""
    keep = torch.ones(env.n_envs, dtype=torch.bool, device=env.device)
    keep[ids.long()] = False
    for k, v in snap.items():
        t = getattr(env, k)
        if k == "agent_pos":
            t[:, keep] = v[:, keep]
        elif t.shape[0] == env.n_envs:     # not the shared [1, K, 2] targets
            t[keep] = v[keep]


def _with_rows(env, ids, acts, g):
    """A full action batch whose rows ids[j] are acts[j] (the others random)."""
    full = _actions(env, env.n_envs, g)
    wide = full.to(torch.int64) if full.dtype == torch.uint16 else full     # no uint16 indexing kernels
    wide[ids.long()] = acts.to(wide.dtype)
    return wide.to(full.dtype)


def _twin_step(twin, ids, acts, agent, g):
    """What a subset step should do, built from a full step: B's unlisted rows go back to their pre-step values."""
    snap = _snapshot(twin)
    twin.step(_with_rows(twin, ids, acts, g), agent=agent)
    _restore_unlisted(twin, snap, ids)


def _env(case, **kw):
    cfg = P.make_config(case.problem, case.rep, map_shape=case.shape, **case.cfg)
    return P.BatchedPcgrlEnv(cfg, case.n, seed=3, **dict(case.env, **kw))


def _twin_of(env, case, **kw):
    """A twin in env's state (state_dict plus the last step's outputs); kw: other constructor options."""
    twin = _env(case, **kw)
    twin.load_state_dict(env.state_dict())
    for k in ("reward", "done", "changed"):
        getattr(twin, k).copy_(getattr(env, k))
    return twin


def _distinct(n, m, rng, dev):
    return torch.from_numpy(rng.permutation(n)[:m].astype(np.int32)).to(dev)


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_step_envs_matches_twin(case):
    env = _make(case)
    g = torch.Generator(device=env.device).manual_seed(17)
    _prepare(env, case, g)
    n = env.n_envs
    rng = np.random.default_rng(5)
    ids = _distinct(n, max(1, 2 * n // 3), rng, env.device)
    acts = _actions(env, ids.numel(), g)
    twin = _twin_of(env, case)
    reward, done = env.step(acts, env_ids=ids, agent=case.agent)
    env.check_status()
    _twin_step(twin, ids, acts, case.agent, g)
    twin.check_status()
    _assert_same(env, twin, case.id)
    assert torch.equal(reward.view(torch.int32), twin.reward[ids.long()].view(torch.int32))
    assert torch.equal(done, twin.done[ids.long()])
    if bool((ids % 4 == 0).any()):                 # _prepare left every fourth env one iteration from done
        assert int(done.sum()) > 0
    assert int(env.changed[ids.long()].sum()) > 0 or case.rep == "cellular"

    # identical full steps afterwards
    for _ in range(3):
        for a in range(max(env.n_agents, 1)):
            acts_s = _actions(env, n, g)
            env.step(acts_s, agent=a)
            twin.step(acts_s, agent=a)
            _assert_same(env, twin, case.id + " after")
    env.check_status()


SEQ_CASES = [c for c in CASES if c.id in ("binary_narrow16", "binary_wide16", "binary_narrow16_fused", "zelda_turtle",
                                          "binary_holey", "binary_patch", "binary_cellular", "sokoban_narrow",
                                          "smb_small", "minecraft_3D_holey_maze", "zelda_turtle_2agents",
                                          "binary_budget", "binary_u8")]


@pytest.mark.parametrize("case", SEQ_CASES, ids=[c.id for c in SEQ_CASES])
def test_step_envs_sequence_with_auto_reset(case):
    """Subset steps (M = 0, 1, N and others, in a random order) across episode ends with auto_reset, mixed with full
    steps, lookahead and observe.  The twin runs without auto_reset and resets the same envs by hand."""
    env = _env(case, auto_reset=True)
    env.reset()
    if env.ctrl_metrics:
        env.sample_uniform_targets(torch.Generator(device=env.device).manual_seed(3))
    g = torch.Generator(device=env.device).manual_seed(23)
    _prepare(env, case, g, steps=3)
    twin = _twin_of(env, case, auto_reset=False)
    n = env.n_envs
    rng = np.random.default_rng(11)
    agents = max(env.n_agents, 1)
    sizes = [0, 1, n] + [int(m) for m in rng.integers(1, n + 1, 9)]
    ops = [("sub", m) for m in sizes] + [("full", 0)] * 3 + [("look", 0), ("obs", 0)] * 2
    finished = 0
    for i in rng.permutation(len(ops)):
        op, m = ops[i]
        a = int(rng.integers(0, agents))
        if op == "sub":
            ids = _distinct(n, m, rng, env.device)
            acts = _actions(env, m, g)
            reward, done = env.step(acts, env_ids=ids.cpu().numpy(), agent=a)
            assert reward.shape == (m,) and done.shape == (m,)
            if m == 0:
                continue
            _twin_step(twin, ids, acts, a, g)
            assert torch.equal(reward.view(torch.int32), twin.reward[ids.long()].view(torch.int32))
            assert torch.equal(done, twin.done[ids.long()])
            mask = torch.zeros(n, dtype=torch.uint8, device=env.device)
            mask[ids.long()] = done
            twin.reset(mask=mask)
            finished += int(done.sum())
            assert env._synced_steps is None
        elif op == "full":
            acts = _actions(env, n, g)
            env.step(acts, agent=a)
            twin.step(acts, agent=a)
            finished += int(twin.done.sum())
            twin.reset(mask=twin.done)
        elif op == "look":
            ids = _distinct(n, n, rng, env.device)
            acts = _actions(env, n, g)
            for x, y in zip(env.lookahead(acts, env_ids=ids, agent=a), twin.lookahead(acts, env_ids=ids, agent=a)):
                assert torch.equal(_bits(x), _bits(y)), case.id
        else:
            ids = _distinct(n, max(1, n // 2), rng, env.device)
            assert torch.equal(env.observe(agent=a, env_ids=ids), twin.observe(agent=a, env_ids=ids))
            assert torch.equal(env.observe(agent=a), twin.observe(agent=a))
        _assert_same(env, twin, f"{case.id} {op} {m}")
        assert env._epoch == twin._epoch
    env.check_status()
    twin.check_status()
    assert finished > 0


def test_step_envs_large_shard():
    """binary narrow 16x16 at 384 Ki envs, two thirds of them listed: many CTAs and a long work list."""
    case = CASES[0]
    n = 384 << 10
    cfg = P.make_config(case.problem, case.rep, map_shape=case.shape)
    env = P.BatchedPcgrlEnv(cfg, n, seed=3)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(29)
    for _ in range(3):
        env.step(_actions(env, n, g))
    env.iteration[::5] = env.max_iterations
    twin = P.BatchedPcgrlEnv(cfg, n, seed=3)
    twin.load_state_dict(env.state_dict())
    for k in ("reward", "done", "changed"):
        getattr(twin, k).copy_(getattr(env, k))
    ids = torch.randperm(n, generator=g, device=env.device)[:2 * n // 3].to(torch.int32)
    for _ in range(2):
        acts = _actions(env, ids.numel(), g)
        reward, _ = env.step(acts, env_ids=ids)
        _twin_step(twin, ids, acts, 0, g)
        _assert_same(env, twin, "large")
        assert torch.equal(reward.view(torch.int32), twin.reward[ids.long()].view(torch.int32))
        acts = _actions(env, n, g)
        env.step(acts)
        twin.step(acts)
        _assert_same(env, twin, "large, full step after")
    env.check_status()


def test_step_envs_validation_before_launch():
    lib = P._lib.load()
    env = _make(CASES[0])
    n = env.n_envs
    z = lambda m: torch.zeros(m, dtype=torch.int32, device=env.device)   # noqa: E731
    torch.cuda.synchronize()
    l0 = lib.pcgrl_launch_count()
    for ids in ([0, n], [-1], torch.tensor([3, n], device=env.device), torch.tensor([-2, 0])):
        with pytest.raises(IndexError):
            env.step(z(len(ids)), env_ids=ids)
    for ids in ([1, 4, 1], np.array([2, 2]), torch.tensor([5, 0, 5], device=env.device),
                torch.tensor([7, 7], dtype=torch.uint8)):
        with pytest.raises(ValueError):
            env.step(z(len(ids)), env_ids=ids)
    with pytest.raises(ValueError):
        env.step(z(3), env_ids=[0, 1])                  # 3 action rows for 2 envs
    with pytest.raises(IndexError):
        env.step(z(1), env_ids=[0], agent=1)            # a single-agent env
    r, d = env.step(z(0), env_ids=[])                   # nothing to step, nothing launched
    assert r.shape == (0,) and d.shape == (0,)
    torch.cuda.synchronize()
    assert lib.pcgrl_launch_count() == l0
    env.update(z(n))
    with pytest.raises(RuntimeError):
        env.step(z(2), env_ids=[0, 1])                  # stale stats
    torch.cuda.synchronize()
    assert lib.pcgrl_launch_count() == l0 + 1           # the update


@pytest.mark.parametrize("case", [CASES[0], CASES[3], CASES[13]], ids=lambda c: c.id)   # indexed, generic x 2
def test_step_envs_device_index_guard(case):
    """An index the host never checked (== n_envs) loads and writes nothing, and sets status bit 256."""
    env = _make(case)
    g = torch.Generator(device=env.device).manual_seed(3)
    _prepare(env, case, g, steps=2)
    lib = P._lib.load()
    snap = _snapshot(env)
    twin = _twin_of(env, case)
    rows = torch.tensor([1, env.n_envs], dtype=torch.int32, device=env.device)
    acts = _actions(env, 2, g)
    work = env._work(int(lib.pcgrl_step_envs_work_bytes(env._cc, 2)))
    P._lib.check(lib.pcgrl_step_envs(env._cc, env._st, acts.data_ptr(), rows.data_ptr(), 2, work.data_ptr(),
                                     env._stream()), "pcgrl_step_envs")
    with pytest.raises(IndexError):
        env.check_status()
    _twin_step(twin, rows[:1], acts[:1], 0, g)
    _assert_same(env, twin, case.id)
    assert not torch.equal(env.iteration, snap["iteration"])
