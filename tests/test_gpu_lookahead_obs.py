"""One-step lookahead with the observation (pcgrl_lookahead_obs, BatchedPcgrlEnv.lookahead(obs_dtype=...) and
lookahead_all(obs_dtype=...)) against a twin env that really takes the step.

The twin: the candidates' envs are saved from the env and loaded into a second env with one slot per candidate, which
steps every slot with its candidate's action (step(env_ids=...)) and observes them with the same options.  For every
config of tests/test_gpu_lookahead.py, after a few random steps (some envs one iteration or one change from done):
  - the observation equals the twin's, byte for byte, as uint8 / float32 / float64 one-hot and as tile codes;
  - reward, done, changed and stats equal lookahead() without the observation and the twin's;
  - the env is untouched: save_envs() before and after are byte-identical, and so is observe().
Then: the incremental path against the same shard without a search cache, invalid actions, multi-agent turtle with
the agent-occupancy plane, a batch large enough for two trips of every CTA of the observation writer, and the checks
before any launch."""
import numpy as np
import pytest
import torch

import control_pcgrl_b200 as P
from tests.test_gpu_lookahead import CASES, Case, _actions, _make, _prepare

pytestmark = pytest.mark.gpu

KINDS = ((torch.uint8, True), (torch.float32, True), (torch.float64, True), (torch.uint8, False))


def _kinds(env):
    # target planes are fractional: no uint8 observation with controls
    return [k for k in KINDS if not (env.ctrl_metrics and k[0] == torch.uint8)]


def _twin(env, case, env_ids, acts, agent):
    """A twin whose slot j is env env_ids[j] after it took action row j: -> (twin, reward, done, stats, changed)."""
    m = env_ids.numel()
    cfg = P.make_config(case.problem, case.rep, map_shape=case.shape, **case.cfg)
    twin = P.BatchedPcgrlEnv(cfg, m, seed=11, **case.env)
    twin.reset()
    twin.load_envs(env.save_envs(env_ids))
    slots = torch.arange(m, dtype=torch.int32, device=env.device)
    reward, done = twin.step(acts, env_ids=slots, agent=agent)
    return twin, reward, done, twin.stats.clone(), twin.changed.clone()


def _assert_outputs(got, want, what):
    for name, a, b in zip(("reward", "done", "stats", "changed"), got, want):
        if name == "reward":   # bit for bit
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (what, name)
        else:
            assert torch.equal(a, b), (what, name)


def _check_against_twin(env, case, env_ids, acts, agent, kinds, pass_ids=True):
    twin, *want = _twin(env, case, env_ids, acts, agent)
    twin.check_status()
    for dtype, onehot in kinds:
        got = env.lookahead(acts, env_ids=env_ids if pass_ids else None, agent=agent, obs_dtype=dtype, onehot=onehot)
        what = f"{case.id} {dtype} onehot={onehot}"
        _assert_outputs(got[:4], want, what)
        _assert_outputs(got[:4], env.lookahead(acts, env_ids=env_ids if pass_ids else None, agent=agent), what)
        ref = twin.observe(dtype=dtype, onehot=onehot, agent=agent)
        assert got[4].dtype == ref.dtype and got[4].shape == ref.shape, what
        assert torch.equal(got[4], ref), what
    return want


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_lookahead_obs_matches_twin(case):
    env = _make(case)
    g = torch.Generator(device=env.device).manual_seed(17)
    _prepare(env, case, g)
    n = env.n_envs
    env_ids = torch.from_numpy(np.random.default_rng(5).integers(0, n, 3 * n).astype(np.int32)).to(env.device)
    acts = _actions(env, env_ids.numel(), g)
    rows0 = env.save_envs()
    obs0 = env.observe(dtype=torch.float32)
    want = _check_against_twin(env, case, env_ids, acts, case.agent, _kinds(env))
    assert bool(want[1].any())                              # some candidates end the episode: terminal observations
    assert torch.equal(env.save_envs(), rows0)              # the shard is untouched
    assert torch.equal(env.observe(dtype=torch.float32), obs0)
    env.check_status()
    # env_ids=None: candidate j is env j
    acts_n = _actions(env, n, g)
    _check_against_twin(env, case, torch.arange(n, dtype=torch.int32, device=env.device), acts_n, case.agent,
                        _kinds(env)[1:2], pass_ids=False)
    assert torch.equal(env.save_envs(), rows0)
    # lookahead_all: column a is lookahead() of action a
    if env.action_kind in ("int32", "wide_flat"):
        A = env.n_discrete_actions()
        ids = np.array([n - 1, 0, n // 2, 0])
        dtype = torch.float32
        all_ = env.lookahead_all(env_ids=ids, agent=case.agent, obs_dtype=dtype)
        assert all_[4].shape == (len(ids), A, *env.obs_shape())
        for a in range(A):
            col = env.lookahead(torch.full((len(ids),), a, device=env.device).to(env._action_layout()[2]), env_ids=ids,
                                agent=case.agent, obs_dtype=dtype)
            _assert_outputs(tuple(t[:, a] for t in all_[:4]), col[:4], f"{case.id} column {a}")
            assert torch.equal(all_[4][:, a], col[4]), f"{case.id} column {a}"
        assert torch.equal(env.save_envs(), rows0)


SHOW_AGENTS = Case("zelda_turtle_3agents_show", "zelda", "turtle", (7, 11), cfg=dict(show_agents=True),
                   env=dict(n_agents=3), agent=2)


@pytest.mark.parametrize("agent", [1, 2])
def test_multiagent_show_agents(agent):
    """The occupancy plane: every agent of env e where it stands, the acting agent where the candidate moves it."""
    env = _make(SHOW_AGENTS)
    assert env.show_agents
    g = torch.Generator(device=env.device).manual_seed(3)
    _prepare(env, SHOW_AGENTS, g)
    n = env.n_envs
    env_ids = torch.from_numpy(np.random.default_rng(1).integers(0, n, 4 * n).astype(np.int32)).to(env.device)
    acts = torch.from_numpy(np.random.default_rng(2).integers(0, 4 + env.n_tiles, 4 * n).astype(np.int32)).to(env.device)
    acts[:8] = torch.tensor([0, 1, 2, 3, 0, 1, 2, 3], dtype=torch.int32)     # moves, some against the edge
    rows0 = env.save_envs()
    _check_against_twin(env, SHOW_AGENTS, env_ids, acts, agent, _kinds(env))
    # obs_out, which receives the occupancy plane too
    out = torch.full((4 * n, *env.obs_shape()), 7, dtype=torch.float32, device=env.device)
    got = env.lookahead(acts, env_ids=env_ids, agent=agent, obs_out=out)
    assert got[4].data_ptr() == out.data_ptr()
    assert torch.equal(out, _twin(env, SHOW_AGENTS, env_ids, acts, agent)[0].observe(agent=agent))
    all_ = env.lookahead_all(env_ids=[0, n - 1], agent=agent, obs_dtype=torch.float32)
    for a in range(env.n_discrete_actions()):
        col = env.lookahead(torch.full((2,), a, dtype=torch.int32, device=env.device), env_ids=[0, n - 1], agent=agent,
                            obs_dtype=torch.float32)
        assert torch.equal(all_[4][:, a], col[4])
    assert torch.equal(env.save_envs(), rows0)


@pytest.mark.parametrize("rep", ["narrow", "turtle", "wide"])
def test_incremental_and_generic_paths_agree(rep):
    """The same 16x16 states with and without a search cache give the same outputs and observations."""
    lib = P._lib.load()
    kw = dict(obs_window=(16, 16)) if rep == "wide" else {}
    cfg = P.make_config("binary", rep, map_shape=(16, 16), controls=["regions", "path-length"], **kw)
    n = 64
    inc, gen = (P.BatchedPcgrlEnv(cfg, n, seed=9, split_step=s) for s in (True, False))
    grids = (np.random.default_rng(2).random((n, 16, 16)) < 0.5).astype(np.int8)
    pos = np.random.default_rng(3).integers(0, 16, (n, 2))
    for e in (inc, gen):
        e.reset(grids=grids, pos=pos if rep == "turtle" else None)
        e.sample_uniform_targets(torch.Generator(device=e.device).manual_seed(4))
    g = torch.Generator(device=inc.device).manual_seed(4)
    for _ in range(6):
        a = _actions(inc, n, g)
        inc.step(a)
        gen.step(a)
    assert torch.equal(inc.stats, gen.stats) and torch.equal(inc.grids, gen.grids)
    assert inc.cache is not None and gen.cache is None
    out = []
    for e, launches in ((inc, 6), (gen, 3)):   # gather, 3 incremental, apply, observe / gather, step, observe
        torch.cuda.synchronize()
        l0 = lib.pcgrl_launch_count()
        r = e.lookahead_all(obs_dtype=torch.float32)
        torch.cuda.synchronize()
        assert lib.pcgrl_launch_count() - l0 == launches, (rep, e.cache is not None)
        out.append(r)
    _assert_outputs(out[0][:4], out[1][:4], rep)
    assert torch.equal(out[0][4], out[1][4]), rep


def test_invalid_actions_and_frozen_cells():
    """Out-of-range actions change nothing but status bit 0, as the step; edits of frozen cells are undone."""
    for case in (next(c for c in CASES if c.id == "binary_static"), next(c for c in CASES if c.id == "zelda_turtle_static")):
        env = _make(case)
        g = torch.Generator(device=env.device).manual_seed(5)
        _prepare(env, case, g)
        n = env.n_envs
        env_ids = torch.arange(n, dtype=torch.int32, device=env.device).repeat(2)
        acts = _actions(env, 2 * n, g)
        acts[::3] = env.n_discrete_actions() + 3                                # invalid
        assert env.static_mask is not None and bool(env.static_mask.any())
        twin, *want = _twin(env, case, env_ids, acts, 0)
        with pytest.raises(ValueError):
            twin.check_status()
        got = env.lookahead(acts, env_ids=env_ids, obs_dtype=torch.float32)
        with pytest.raises(ValueError):
            env.check_status()
        _assert_outputs(got[:4], want, case.id)
        assert torch.equal(got[4], twin.observe())


def test_two_trips_of_the_observation_writer():
    """40000 candidates: the writer's grid is at most 148 SMs x 8 CTAs of 256 threads, each holding at most 8 envs
    of the binary u8 32x32x3 crop (fewer in float32), so every CTA makes at least two trips."""
    for case in (CASES[0], next(c for c in CASES if c.id == "zelda_turtle")):    # incremental, generic
        env = _make(case, seed=4)
        g = torch.Generator(device=env.device).manual_seed(6)
        _prepare(env, case, g)
        n, A = env.n_envs, env.n_discrete_actions()
        rows0 = env.save_envs()
        ref = {}
        for dtype in (torch.uint8, torch.float32):
            # every (env, action) pair once, against the twin
            pairs = torch.arange(n * A, dtype=torch.int32, device=env.device)
            twin = _twin(env, case, pairs // A, (pairs % A).to(torch.int32), 0)[0]
            ref[dtype] = twin.observe(dtype=dtype).view(n, A, *env.obs_shape())
            assert torch.equal(env.lookahead_all(obs_dtype=dtype)[4], ref[dtype])
        m = 40000
        rng = np.random.default_rng(7)
        e = torch.from_numpy(rng.integers(0, n, m).astype(np.int32)).to(env.device)
        a = torch.from_numpy(rng.integers(0, A, m).astype(np.int32)).to(env.device)
        for dtype in (torch.uint8, torch.float32):
            got = env.lookahead(a, env_ids=e, obs_dtype=dtype)[4]
            assert torch.equal(got, ref[dtype][e.long(), a.long()]), (case.id, dtype)
        assert torch.equal(env.save_envs(), rows0)
        env.check_status()


def test_lookahead_all_bounds_the_observation_bytes_per_launch(monkeypatch):
    env = _make(CASES[0])
    g = torch.Generator(device=env.device).manual_seed(2)
    _prepare(env, CASES[0], g)
    lib = P._lib.load()
    whole = env.lookahead_all(obs_dtype=torch.uint8)
    # three envs' observations per launch: 24 envs -> 8 launches of 6 (gather, 3 incremental, apply, observe) each
    monkeypatch.setattr(env, "LOOKAHEAD_OBS_CHUNK_BYTES", 3 * env.n_discrete_actions() * int(np.prod(env.obs_shape())))
    torch.cuda.synchronize()
    l0 = lib.pcgrl_launch_count()
    chunked = env.lookahead_all(obs_dtype=torch.uint8)
    torch.cuda.synchronize()
    assert lib.pcgrl_launch_count() - l0 == 6 * (env.n_envs // 3)
    for a, b in zip(whole, chunked):
        assert torch.equal(a, b)


def test_validation_before_any_launch():
    lib = P._lib.load()
    env = _make(CASES[0])
    env.step(torch.zeros(env.n_envs, dtype=torch.int32, device=env.device))
    ctrl = _make(next(c for c in CASES if c.id == "binary_controls"))
    z = torch.zeros(2, dtype=torch.int32, device=env.device)
    torch.cuda.synchronize()
    l0 = lib.pcgrl_launch_count()
    for ids in ([0, env.n_envs], [-1], torch.tensor([0, env.n_envs], device=env.device)):
        with pytest.raises(IndexError):
            env.lookahead(z[:len(ids)], env_ids=ids, obs_dtype=torch.uint8)
        with pytest.raises(IndexError):
            env.lookahead_all(env_ids=ids, obs_dtype=torch.uint8)
    shape = (2, *env.obs_shape())
    for bad in (torch.empty((3, *shape[1:]), dtype=torch.uint8, device=env.device),
                torch.empty((*shape[:-1], shape[-1] + 1), dtype=torch.uint8, device=env.device),
                torch.empty((2, shape[2], shape[1], shape[3]), dtype=torch.uint8, device=env.device).transpose(1, 2)):
        with pytest.raises(ValueError):
            env.lookahead(z, env_ids=[0, 1], obs_out=bad)
    with pytest.raises(ValueError):   # tile codes are uint8
        env.lookahead(z, env_ids=[0, 1], obs_out=torch.empty(shape[:-1] + (1,), device=env.device), onehot=False)
    with pytest.raises(ValueError):   # target planes are fractional
        ctrl.lookahead(z, env_ids=[0, 1], obs_dtype=torch.uint8, onehot=False)
    # n = 0: empty tensors, nothing launched
    r = env.lookahead(z[:0], env_ids=[], obs_dtype=torch.float32)
    assert r[0].shape == (0,) and r[4].shape == (0, *env.obs_shape())
    r = env.lookahead_all(env_ids=np.zeros(0, dtype=np.int64), obs_dtype=torch.float32)
    assert r[4].shape == (0, 2, *env.obs_shape())
    torch.cuda.synchronize()
    assert lib.pcgrl_launch_count() == l0
    # stale stats after update()
    env.update(torch.ones(env.n_envs, dtype=torch.int32, device=env.device))
    torch.cuda.synchronize()
    l0 = lib.pcgrl_launch_count()
    with pytest.raises(RuntimeError):
        env.lookahead(torch.zeros(env.n_envs, dtype=torch.int32, device=env.device), obs_dtype=torch.float32)
    with pytest.raises(RuntimeError):
        env.lookahead_all(obs_dtype=torch.float32)
    assert lib.pcgrl_launch_count() == l0


def test_device_index_guard():
    """A device index the host never checked loads nothing and sets status bit 128; the shard is untouched."""
    for case in (CASES[0], next(c for c in CASES if c.id == "zelda_narrow")):    # incremental, generic
        env = _make(case)
        rows0 = env.save_envs()
        rows = torch.tensor([0, env.n_envs + 5], dtype=torch.int32, device=env.device)
        a = torch.zeros(2, dtype=torch.int32, device=env.device)
        outs = (torch.empty(2, dtype=torch.float32, device=env.device), torch.empty(2, dtype=torch.uint8, device=env.device),
                torch.empty((2, env.K), dtype=torch.int32, device=env.device),
                torch.empty(2, dtype=torch.uint8, device=env.device))
        obs = env._lookahead_obs(a, rows, 2, 0, outs, None, torch.float32, True)
        torch.cuda.synchronize()
        assert torch.equal(env.save_envs(), rows0)
        with pytest.raises(IndexError):
            env.check_status()
        good = env.lookahead(a[:1], env_ids=[0], obs_dtype=torch.float32)
        assert torch.equal(obs[:1], good[4]) and torch.equal(outs[2][:1], good[2])
