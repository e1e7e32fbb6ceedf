"""One-step lookahead (pcgrl_lookahead, BatchedPcgrlEnv.lookahead / lookahead_all) against a twin env stepped by hand.

For every config below, after a few random steps (and a masked reset, so that positions and counters differ, with
some envs one iteration or one change from done):
  - random candidates (any order, duplicates) match what a twin restored from state_dict() returns when it steps the
    same env with the same action -- reward bit for bit, done, changed and the stats row.  The candidates are run in
    rounds in which every env appears at most once, one twin step per round;
  - every state tensor of the env, and the last step's outputs, are bitwise unchanged by the lookahead;
  - afterwards the env and a twin that never looked ahead agree at every step of the same actions (hidden work-list
    or scratch state would show here);
  - lookahead_all equals lookahead column by column (Discrete action spaces).
Then: the incremental and generic paths agree on the same 16x16 states, invalid actions and env indices, empty and
bad env_ids, stale stats, and lookahead_all without a host sync."""
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch

import control_pcgrl_b200 as P

pytestmark = pytest.mark.gpu


@dataclass
class Case:
    id: str
    problem: str
    rep: str
    shape: tuple
    n: int = 24
    cfg: dict = field(default_factory=dict)
    env: dict = field(default_factory=dict)
    agent: int = 0
    inc: bool = False          # the shard has a search cache: the incremental path


CASES = [
    Case("binary_narrow16", "binary", "narrow", (16, 16), inc=True),
    Case("binary_turtle16", "binary", "turtle", (16, 16), inc=True),
    Case("binary_wide16", "binary", "wide", (16, 16), cfg=dict(obs_window=(16, 16)), inc=True),
    Case("binary_narrow16_fused", "binary", "narrow", (16, 16), env=dict(split_step=False)),
    Case("binary_narrow32", "binary", "narrow", (32, 32)),
    Case("binary_narrow64", "binary", "narrow", (64, 64), n=8),
    Case("zelda_narrow", "zelda", "narrow", (7, 11)),
    Case("zelda_turtle", "zelda", "turtle", (7, 11)),
    Case("binary_holey", "binary_holey", "narrow", (16, 16)),
    Case("minecraft_2D_maze", "minecraft_2D_maze", "narrow", (14, 14), inc=True),
    Case("binary_static", "binary", "narrow", (16, 16), cfg=dict(static_tile_wrapper=True, static_prob=0.6,
                                                                  n_static_walls=2), inc=True),
    Case("zelda_turtle_static", "zelda", "turtle", (7, 11), cfg=dict(static_tile_wrapper=True, static_prob=0.6)),
    Case("binary_patch", "binary", "narrow", (16, 16), cfg=dict(act_window=(3, 3))),
    Case("binary_cellular", "binary", "cellular", (16, 16)),
    Case("sokoban_cellular", "sokoban", "cellular", (5, 5), env=dict(action_kind="ca_tiles")),
    Case("sokoban_narrow", "sokoban", "narrow", (5, 5)),
    Case("smb_small", "smb", "narrow", (12, 10), n=8),
    Case("minecraft_3D_maze", "minecraft_3D_maze", "narrow", (14, 14, 14), n=6),
    Case("minecraft_3D_holey_maze", "minecraft_3D_holey_maze", "narrow", (14, 14, 14), n=6),
    Case("zelda_turtle_2agents", "zelda", "turtle", (7, 11), env=dict(n_agents=2), agent=1),
    Case("binary_budget", "binary", "narrow", (16, 16), cfg=dict(change_percentage=0.05), inc=True),
    Case("zelda_budget", "zelda", "turtle", (7, 11), cfg=dict(change_percentage=0.1)),
    Case("binary_controls", "binary", "narrow", (16, 16), cfg=dict(controls=["regions", "path-length"]), inc=True),
    Case("zelda_controls", "zelda", "narrow", (7, 11), cfg=dict(controls=["regions", "path-length", "enemies"])),
    Case("binary_range", "binary", "narrow", (16, 16), env=dict(reward_mode="range"), inc=True),
    Case("binary_u8", "binary", "narrow", (16, 16), env=dict(compact_host_io=True), inc=True),
    Case("binary_wide_u8", "binary", "wide", (16, 16), cfg=dict(obs_window=(16, 16)), env=dict(compact_host_io=True),
         inc=True),
    Case("zelda_turtle_u8", "zelda", "turtle", (7, 11), env=dict(compact_host_io=True)),
]

STATE = ("grids", "agent_pos", "n_step", "iteration", "changes", "stats", "targets", "reward", "done", "changed",
         "records", "cache", "static_mask", "holes", "scratch", "worklist")


def _make(case, seed=3):
    cfg = P.make_config(case.problem, case.rep, map_shape=case.shape, **case.cfg)
    env = P.BatchedPcgrlEnv(cfg, case.n, seed=seed, **case.env)
    env.reset()
    if env.ctrl_metrics:
        env.sample_uniform_targets(torch.Generator(device=env.device).manual_seed(seed))
    return env


def _actions(env, m, g):
    """m random valid actions in env's layout (a device generator: no host sync)."""
    shape, _, tdt = env._action_layout(m)
    dev = env.device
    k = env.action_kind
    if k in ("int32", "wide_flat"):
        a = torch.randint(0, env.n_discrete_actions(), (m,), generator=g, device=dev)
    elif k == "wide_coords":
        cols = [torch.randint(0, d, (m,), generator=g, device=dev) for d in env.map_shape]
        a = torch.stack(cols + [torch.randint(0, env.n_tiles, (m,), generator=g, device=dev)], 1)
    elif k == "patch":
        a = torch.randint(0, env.n_tiles, shape, generator=g, device=dev)
    elif k == "ca_tiles":
        a = torch.zeros(shape, dtype=torch.int64, device=dev)
        a[:, :env.cells] = torch.randint(0, env.n_tiles, (m, env.cells), generator=g, device=dev)
    else:
        a = torch.randn(shape, generator=g, device=dev)
    return a.to(tdt).reshape(shape).contiguous()


def _prepare(env, case, g, steps=5):
    """A few steps, a masked reset, more steps, then some envs one iteration / one change from done."""
    agents = range(max(env.n_agents, 1))
    for t in range(steps):
        for a in agents:
            env.step(_actions(env, env.n_envs, g), agent=a)
        if t == 1:
            env.reset(mask=(torch.arange(env.n_envs, device=env.device) % 3 == 0).to(torch.uint8))
    env.iteration[::4] = env.max_iterations
    if env.max_changes is not None:
        env.changes[1::4] = env.max_changes
    env.check_status()


def _snapshot(env):
    return {k: getattr(env, k).clone() for k in STATE if getattr(env, k) is not None}


def _assert_unchanged(env, snap, what):
    for k, v in snap.items():   # bytewise: targets hold NaN
        assert torch.equal(getattr(env, k).reshape(-1).view(torch.uint8), v.reshape(-1).view(torch.uint8)), (what, k)


def _rounds(env_ids):
    """Split candidate positions into rounds in which every env appears at most once."""
    seen, rounds = {}, []
    for j, e in enumerate(env_ids.tolist()):
        r = seen.get(e, 0)
        seen[e] = r + 1
        if r == len(rounds):
            rounds.append([])
        rounds[r].append(j)
    return rounds


def _twin_outputs(case, sd, acts, env_ids, agent, g):
    """What a twin restored from sd returns for each candidate, one step per round."""
    twin = _make(case)
    m = env_ids.numel()
    K = twin.K
    reward = torch.empty(m, dtype=torch.float32, device=twin.device)
    done = torch.empty(m, dtype=torch.uint8, device=twin.device)
    changed = torch.empty(m, dtype=torch.uint8, device=twin.device)
    stats = torch.empty((m, K), dtype=torch.int32, device=twin.device)
    for rnd in _rounds(env_ids):
        twin.load_state_dict(sd)
        full = _actions(twin, twin.n_envs, g)
        j = torch.tensor(rnd, device=twin.device)
        e = env_ids[j].long()
        wide = full.to(torch.int64) if full.dtype == torch.uint16 else full    # no uint16 indexing kernels
        wide[e] = acts.to(wide.dtype)[j]
        twin.step(wide.to(full.dtype), agent=agent)
        reward[j], done[j], changed[j], stats[j] = twin.reward[e], twin.done[e], twin.changed[e], twin.stats[e]
    twin.check_status()
    return reward, done, stats, changed


def _assert_equal_outputs(got, want, what):
    for name, a, b in zip(("reward", "done", "stats", "changed"), got, want):
        if name == "reward":   # bit for bit
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (what, name, a, b)
        else:
            assert torch.equal(a, b), (what, name)


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_lookahead_matches_twin(case):
    env = _make(case)
    g = torch.Generator(device=env.device).manual_seed(17)
    _prepare(env, case, g)
    assert (env.cache is not None) == case.inc
    sd = env.state_dict()
    n = env.n_envs
    rng = np.random.default_rng(5)
    env_ids = torch.from_numpy(rng.integers(0, n, 3 * n).astype(np.int32)).to(env.device)
    acts = _actions(env, env_ids.numel(), g)
    snap = _snapshot(env)
    got = env.lookahead(acts, env_ids=env_ids, agent=case.agent)
    _assert_unchanged(env, snap, "lookahead")
    env.check_status()
    want = _twin_outputs(case, sd, acts, env_ids, case.agent, g)
    _assert_equal_outputs(got, want, case.id)
    assert 0 < int(got[3].sum()) or case.rep == "cellular"

    # env_ids=None: candidate j is env j
    acts_n = _actions(env, n, g)
    got_n = env.lookahead(acts_n, agent=case.agent)
    _assert_unchanged(env, snap, "lookahead env_ids=None")
    _assert_equal_outputs(got_n, _twin_outputs(case, sd, acts_n, torch.arange(n, device=env.device, dtype=torch.int32),
                                               case.agent, g), case.id + " env_ids=None")

    # the env and a twin that never looked ahead agree at every later step
    twin = _make(case)
    twin.load_state_dict(sd)
    for _ in range(4):
        for a in range(max(env.n_agents, 1)):
            acts_s = _actions(env, n, g)
            r1, d1 = env.step(acts_s, agent=a)
            r2, d2 = twin.step(acts_s, agent=a)
            assert torch.equal(r1.view(torch.int32), r2.view(torch.int32)) and torch.equal(d1, d2)
            assert torch.equal(env.stats, twin.stats) and torch.equal(env.grids, twin.grids)
            assert torch.equal(env.changed, twin.changed)
    env.check_status()

    if env.action_kind in ("int32", "wide_flat"):
        A = env.n_discrete_actions()
        ids = np.array([n - 1, 0, n // 2, 0])
        all_ = env.lookahead_all(env_ids=ids, agent=case.agent)
        for a in range(A):
            col = env.lookahead(torch.full((len(ids),), a, device=env.device).to(env._action_layout()[2]), env_ids=ids,
                                agent=case.agent)
            _assert_equal_outputs(tuple(t[:, a] for t in all_), col, f"{case.id} column {a}")


def test_lookahead_all_current_tile_is_a_no_op():
    """binary narrow: writing the tile that is already there changes nothing: reward 0, the env's own stats."""
    env = _make(CASES[0])
    g = torch.Generator(device=env.device).manual_seed(1)
    _prepare(env, CASES[0], g)
    reward, done, stats, changed = env.lookahead_all()
    pos = env.pos[:, 0] * 16 + env.pos[:, 1]
    cur = env.grids.gather(1, pos[:, None].long())[:, 0].long()
    rows = torch.arange(env.n_envs, device=env.device)
    assert int(changed[rows, cur].sum()) == 0 and int(changed[rows, 1 - cur].min()) == 1
    assert float(reward[rows, cur].abs().max()) == 0.0
    assert torch.equal(stats[rows, cur], env.stats)
    # done: one more iteration, no more change
    assert torch.equal(done[rows, cur].bool(), env.iteration + 1 > env.max_iterations)


@pytest.mark.parametrize("rep", ["narrow", "turtle", "wide"])
def test_incremental_and_generic_paths_agree(rep):
    lib = P._lib.load()
    kw = dict(obs_window=(16, 16)) if rep == "wide" else {}
    cfg = P.make_config("binary", rep, map_shape=(16, 16), **kw)
    n = 64
    inc, gen = (P.BatchedPcgrlEnv(cfg, n, seed=9, split_step=s) for s in (True, False))
    grids = (np.random.default_rng(2).random((n, 16, 16)) < 0.5).astype(np.int8)
    pos = np.random.default_rng(3).integers(0, 16, (n, 2))
    for e in (inc, gen):
        e.reset(grids=grids, pos=pos if rep == "turtle" else None)
    g = torch.Generator(device=inc.device).manual_seed(4)
    for _ in range(6):
        a = _actions(inc, n, g)
        inc.step(a)
        gen.step(a)
    assert torch.equal(inc.stats, gen.stats) and torch.equal(inc.grids, gen.grids)
    assert inc.cache is not None and gen.cache is None
    out = []
    for e, launches in ((inc, 3), (gen, 2)):
        l0 = lib.pcgrl_launch_count()
        r = e.lookahead_all()
        torch.cuda.synchronize()
        assert lib.pcgrl_launch_count() - l0 == launches, (rep, e.cache is not None)
        out.append(r)
    _assert_equal_outputs(out[0], out[1], rep)


def test_invalid_action_and_env_index():
    env = _make(CASES[0])
    env.step(torch.zeros(env.n_envs, dtype=torch.int32, device=env.device))
    bad = torch.full((3,), 7, dtype=torch.int32, device=env.device)
    env.lookahead(bad, env_ids=[0, 1, 2])
    with pytest.raises(ValueError):
        env.check_status()
    env.check_status()
    for ids in ([0, env.n_envs], [-1], torch.tensor([env.n_envs], device=env.device)):
        with pytest.raises(IndexError):
            env.lookahead(torch.zeros(len(ids), dtype=torch.int32, device=env.device), env_ids=ids)
        with pytest.raises(IndexError):
            env.lookahead_all(env_ids=ids)
    # a device index the host never checked: nothing is loaded through it, status bit 128
    for case in (CASES[0], CASES[6]):   # incremental, generic
        e = _make(case)
        snap = _snapshot(e)
        rows = torch.tensor([0, e.n_envs + 5], dtype=torch.int32, device=e.device)
        outs = (torch.empty(2, dtype=torch.float32, device=e.device), torch.empty(2, dtype=torch.uint8, device=e.device),
                torch.empty((2, e.K), dtype=torch.int32, device=e.device), torch.empty(2, dtype=torch.uint8, device=e.device))
        e._lookahead(torch.zeros(2, dtype=torch.int32, device=e.device), rows, 2, 0, *outs)
        _assert_unchanged(e, snap, case.id)
        with pytest.raises(IndexError):
            e.check_status()
    # empty: empty tensors, nothing launched
    lib = P._lib.load()
    torch.cuda.synchronize()
    l0 = lib.pcgrl_launch_count()
    r, d, s, c = env.lookahead(torch.zeros(0, dtype=torch.int32, device=env.device), env_ids=[])
    assert r.shape == (0,) and d.shape == (0,) and s.shape == (0, env.K) and c.shape == (0,)
    r, d, s, c = env.lookahead_all(env_ids=np.zeros(0, dtype=np.int64))
    assert r.shape == (0, 2) and s.shape == (0, 2, env.K)
    assert lib.pcgrl_launch_count() == l0


def test_stale_stats_raise_and_unsupported_spaces():
    env = _make(CASES[0])
    env.update(torch.ones(env.n_envs, dtype=torch.int32, device=env.device))
    with pytest.raises(RuntimeError):
        env.lookahead(torch.zeros(env.n_envs, dtype=torch.int32, device=env.device))
    with pytest.raises(RuntimeError):
        env.lookahead_all()
    for case in (next(c for c in CASES if c.id == "binary_patch"), next(c for c in CASES if c.id == "binary_cellular")):
        with pytest.raises(ValueError):
            _make(case).lookahead_all()
    wc = P.BatchedPcgrlEnv(P.make_config("binary", "wide", map_shape=(16, 16), obs_window=(16, 16)), 4,
                           action_kind="wide_coords")
    wc.reset()
    with pytest.raises(ValueError):
        wc.lookahead_all()
    wide_big = P.BatchedPcgrlEnv(P.make_config("binary", "wide", map_shape=(16, 16)), 4)   # ActionMap 32 x 32
    wide_big.reset()
    with pytest.raises(ValueError):
        wide_big.lookahead_all()


def test_lookahead_all_has_no_host_sync():
    env = _make(CASES[0])
    g = torch.Generator(device=env.device).manual_seed(2)
    _prepare(env, CASES[0], g)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = env.lookahead_all()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert out[0].shape == (env.n_envs, 2)
