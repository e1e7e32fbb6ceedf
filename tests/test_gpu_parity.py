"""GPU parity tests: the CUDA path (through the C ABI) vs the reference-generated fixtures and the oracle.

Bit-exact: grids, stats, positions, done flags, change counters.  Rewards: rel 1e-6 (BASELINE.json).
"""
import numpy as np
import pytest
import torch

from tests.golden_util import TRACES, TRACES_SEARCH, TRACES_WRAPPED, Trace, load_stats

pytestmark = pytest.mark.gpu


def _mk(problem, rep, map_shape, n, **kw):
    import control_pcgrl_b200 as P
    cfg = P.make_config(problem, rep, map_shape=map_shape, **{k: v for k, v in kw.items()
                                                              if k in ("obs_window", "weights", "controls",
                                                                       "max_board_scans", "change_percentage",
                                                                       "act_window", "static_tile_wrapper",
                                                                       "static_prob", "n_static_walls")})
    extra = {k: v for k, v in kw.items() if k in ("action_kind", "auto_reset", "seed", "env_offset")}
    return P.BatchedPcgrlEnv(cfg, n, **extra)


@pytest.mark.parametrize("name,problem", [("binary", "binary"), ("binary_shapes", "binary"), ("zelda", "zelda"),
                                          ("maze3d", "minecraft_3D_maze"), ("sokoban", "sokoban"), ("smb", "smb"),
                                          ("minecraft_2D_maze", "minecraft_2D_maze"),
                                          ("binary_big", "binary"), ("zelda_big", "zelda")])
def test_stats_kernel_matches_reference_fixtures(name, problem):
    _, groups = load_stats(name)
    total = 0
    for grids, stats in groups:
        shape = grids.shape[1:]
        if max(shape) > 64 and problem in ("binary", "zelda"):
            continue
        env = _mk(problem, "narrow", shape, 1)
        got = env.compute_stats(grids).cpu().numpy()
        bad = np.flatnonzero((got != stats).any(axis=1))
        assert bad.size == 0, (name, shape, bad[:5], got[bad[:5]], stats[bad[:5]])
        env.check_status()
        total += len(grids)
    assert total > (15 if name.endswith("_big") else 100)


@pytest.mark.parametrize("problem,rep,shape", [("binary", "narrow", (64, 64)), ("zelda", "turtle", (64, 64)),
                                               ("binary", "wide", (48, 48)), ("zelda", "narrow", (33, 20))])
def test_big_board_rollout(problem, rep, shape):
    """Maps beyond 32x32 (binary_bigger / zelda_bigger, configs/task/*_bigger.yaml:5) run on the warp-per-grid
    boards of step_bigboard.cu: step-by-step properties on the batch, stats recomputed from scratch, and the
    oracle on a few envs."""
    from oracle import pcgrl_oracle as O
    n, n_or, steps = 512, 4, 60
    kw = dict(obs_window=shape) if rep == "wide" else {}
    env = _mk(problem, rep, shape, n, seed=21, **kw)
    env.reset()
    assert env.worklist is None and env.cache is None
    assert torch.equal(env.compute_stats(env.maps), env.stats)
    maps0, pos0 = env.maps.cpu().numpy(), env.pos.cpu().numpy()
    oracles = []
    for e in range(n_or):
        o = O.OracleEnv(problem, rep, shape, weights=dict(env.metric_weights))
        o.reset(maps0[e], pos=pos0[e, :2])
        oracles.append(o)
    n_act = {"narrow": env.n_tiles, "turtle": 4 + env.n_tiles, "wide": shape[0] * shape[1] * env.n_tiles}[rep]
    g = torch.Generator(device=env.device).manual_seed(0)
    prev = env.stats.clone()
    for t in range(steps):
        a = torch.randint(0, n_act, (n,), generator=g, device=env.device, dtype=torch.int32)
        reward, _ = env.step(a)
        ch = env.changed.bool()
        assert torch.equal(env.stats[~ch], prev[~ch]) and float(reward[~ch].abs().max()) == 0.0
        prev = env.stats.clone()
        a_h, r_h, st_h = a.cpu().numpy(), reward.cpu().numpy(), env.stats.cpu().numpy()
        for e, o in enumerate(oracles):
            act = int(a_h[e])
            if rep == "wide":
                act = O.actionmap_unravel(act, shape[0], shape[1], env.n_tiles)
            r, _, _ = o.step(act)
            assert st_h[e].tolist() == O.stats_vector(problem, o.stats), (t, e)
            assert r_h[e] == pytest.approx(float(r), rel=1e-6, abs=1e-7), (t, e)
    assert torch.equal(env.compute_stats(env.maps), env.stats)
    obs = env.observe(dtype=torch.uint8)
    assert int(obs.sum()) == n * int(np.prod(obs.shape[1:-1]))
    env.check_status()


@pytest.mark.parametrize("name", TRACES + TRACES_SEARCH + TRACES_WRAPPED)
def test_trace_replay_matches_reference(name):
    tr = Trace(name)
    n = tr.n_envs
    kind = None
    if tr.rep == "wide":
        kind = "wide_coords" if tr.raw_only else "wide_flat"
    if tr.rep == "cellular":
        kind = "ca_logits"
    env = _mk(tr.problem, tr.rep, tr.map_shape, n, obs_window=tr.obs_window, weights=tr.weights,
              controls=tr.controls, max_board_scans=tr.max_board_scans, change_percentage=tr.change_percentage,
              action_kind=kind, act_window=tr.act_window, static_tile_wrapper=tr.static)
    if tr.target_names:
        env.set_trgs({k: np.array([tr.targets(e)[k] for e in range(n)]) for k in tr.target_names})
    grids0 = np.stack([tr.envs[e]["grid0"] for e in range(n)])
    pos0 = np.stack([tr.envs[e]["pos0"] for e in range(n)])
    static0 = np.stack([tr.envs[e]["static"] for e in range(n)]) if tr.static else None
    env.reset(grids=grids0, pos=pos0 if tr.rep == "turtle" else None, static_tiles=static0)
    if tr.rep == "narrow":
        assert env.pos.cpu().numpy()[:, :len(tr.map_shape)].tolist() == pos0.tolist()
    st0 = env.stats.cpu().numpy()
    for e in range(n):
        assert st0[e].tolist() == [int(v) for v in tr.envs[e]["stats0"]], (name, e)
    T = max(len(tr.envs[e]["rewards"]) for e in range(n))
    shape, dt = env.action_shape_dtype()
    for t in range(T):
        a = np.zeros(shape, dtype=dt)
        live = []
        for e in range(n):
            d = tr.envs[e]
            if t < len(d["rewards"]):
                a[e] = np.asarray(d["actions"][t]).reshape(a[e].shape)
                live.append(e)
        reward, done = env.step(torch.from_numpy(a).to(env.device))
        reward, done = reward.cpu().numpy(), done.cpu().numpy()
        stats, maps, pos = env.stats.cpu().numpy(), env.maps.cpu().numpy(), env.pos.cpu().numpy()
        changes = env.changes.cpu().numpy()
        obs = None
        for e in live:
            d = tr.envs[e]
            assert bool(done[e]) == bool(d["dones"][t]), (name, e, t)
            assert stats[e].tolist() == [int(v) for v in d["stats"][t]], (name, e, t)
            if t in d["grid_at"]:
                assert np.array_equal(maps[e].astype(np.uint8), d["grids"][d["grid_at"][t]]), (name, e, t)
            assert int(changes[e]) == int(d["changes"][t]), (name, e, t)
            assert reward[e] == pytest.approx(float(d["rewards"][t]), rel=1e-6, abs=1e-7), (name, e, t)
            if tr.rep in ("narrow", "turtle"):
                assert pos[e, :len(tr.map_shape)].tolist() == [int(v) for v in d["pos"][t]], (name, e, t)
            if t in d["obs_step"]:
                if obs is None:
                    obs = env.observe(dtype=torch.float64).cpu().numpy()
                want = d["obs"][list(d["obs_step"]).index(t)]
                assert obs[e].shape == want.shape
                np.testing.assert_allclose(obs[e], want, rtol=1e-12, atol=0, err_msg=f"{name} env {e} step {t}")
    env.check_status()


def test_random_grids_vs_oracle():
    from oracle import pcgrl_oracle as O
    rng = np.random.default_rng(2026)
    for problem, shape, ntile, probs in [("binary", (16, 16), 2, None), ("binary", (9, 13), 2, None),
                                         ("binary", (24, 31), 2, None),
                                         ("zelda", (7, 11), 8, [0.58, 0.3, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02]),
                                         ("zelda", (12, 20), 8, [0.7, 0.2, 0.02, 0.02, 0.02, 0.02, 0.01, 0.01])]:
        n = 300
        grids = rng.choice(ntile, size=(n, *shape), p=probs).astype(np.int8)
        if problem == "zelda":   # make a good share of them playable-ish
            for i in range(0, n, 2):
                g = grids[i]
                g[(g == 2) | (g == 3) | (g == 4)] = 0
                cells = rng.choice(g.size, size=3, replace=False)
                for c, t in zip(cells, (2, 3, 4)):
                    g.flat[c] = t
        env = _mk(problem, "narrow", shape, 1)
        got = env.compute_stats(grids).cpu().numpy()
        for i in range(n):
            want = O.stats_vector(problem, O.get_stats(problem, grids[i]))
            assert got[i].tolist() == want, (problem, shape, i)


def test_full_size_properties_binary_narrow():
    """BASELINE config sizes (65 536 envs): size-independent properties instead of a CPU oracle run."""
    n = 65536
    env = _mk("binary", "narrow", (16, 16), n, seed=3)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(0)
    assert torch.equal(env.compute_stats(env.maps), env.stats)          # reset stats == fresh recompute
    prev_stats = env.stats.clone()
    prev_maps = env.maps.clone()
    for t in range(40):
        a = torch.randint(0, 2, (n,), generator=g, device=env.device, dtype=torch.int32)
        reward, done = env.step(a)
        ch = env.changed.bool()
        # unchanged envs keep stats and get exactly zero reward
        assert torch.equal(env.stats[~ch], prev_stats[~ch])
        assert float(reward[~ch].abs().max()) == 0.0
        # exactly one cell differs where changed, none elsewhere
        diff = (env.maps != prev_maps).flatten(1).sum(1)
        assert torch.equal(diff, ch.long())
        assert not bool(done.any())
        prev_stats = env.stats.clone()
        prev_maps = env.maps.clone()
    # incremental path == stats recomputed from scratch on the final maps
    assert torch.equal(env.compute_stats(env.maps), env.stats)
    # reward == loss(new) - loss(old) with static targets regions=1, path-length=136, weights 1
    assert torch.equal(env.iteration, torch.full_like(env.iteration, 40))
    # linear bound: regions <= 128, 0 <= path <= 136
    assert int(env.stats[:, 0].max()) <= 128 and int(env.stats[:, 1].max()) <= 136 and int(env.stats.min()) >= 0


@pytest.mark.parametrize("problem,rep,shape,controls", [
    ("binary", "wide", (16, 16), ["regions", "path-length"]),     # BASELINE config 2 at its stated size
    ("zelda", "turtle", (7, 11), None),                           # BASELINE config 3 at its stated size
])
def test_full_size_properties_configs_2_and_3(problem, rep, shape, controls):
    """65 536 envs of binary-wide + ControlWrapper targets (per-env regions / path-length) and of zelda-turtle:
    size-independent properties on the whole batch plus the oracle on a 256-env sample, step by step (stats and
    maps bit-exact, rewards to 1e-6 of the oracle's fp64 loss difference under the env's own targets)."""
    from oracle import pcgrl_oracle as O
    n, n_or = 65536, 256
    kw = dict(obs_window=shape) if rep == "wide" else {}
    env = _mk(problem, rep, shape, n, seed=9, controls=controls, **kw)
    if controls:
        g0 = torch.Generator(device=env.device).manual_seed(2)
        env.sample_uniform_targets(generator=g0)
    env.reset()
    assert torch.equal(env.compute_stats(env.maps), env.stats)
    sample = np.linspace(0, n - 1, n_or).astype(np.int64)
    maps0, pos0 = env.maps.cpu().numpy(), env.pos.cpu().numpy()
    trg = env.targets.cpu().numpy()
    weights = {k: v for k, v in env.metric_weights.items()}
    oracles = []
    for e in sample:
        o = O.OracleEnv(problem, rep, shape, weights=weights, controls=controls)
        targets = {k: float(trg[e, env.stat_names.index(k), 0]) for k in (controls or [])}
        o.reset(maps0[e], pos=pos0[e, :2], targets=targets)
        oracles.append(o)
    n_act = {"turtle": 4 + env.n_tiles, "wide": shape[0] * shape[1] * env.n_tiles}[rep]
    g = torch.Generator(device=env.device).manual_seed(0)
    prev_stats, prev_maps = env.stats.clone(), env.maps.clone()
    for t in range(48):
        a = torch.randint(0, n_act, (n,), generator=g, device=env.device, dtype=torch.int32)
        reward, done = env.step(a)
        ch = env.changed.bool()
        assert torch.equal(env.stats[~ch], prev_stats[~ch]) and float(reward[~ch].abs().max()) == 0.0
        diff = (env.maps != prev_maps).flatten(1).sum(1)
        assert torch.equal(diff, ch.long())                       # one cell per changed env, none elsewhere
        assert not bool(done.any())
        prev_stats, prev_maps = env.stats.clone(), env.maps.clone()
        a_h, r_h, st_h, maps_h = a.cpu().numpy(), reward.cpu().numpy(), env.stats.cpu().numpy(), env.maps.cpu().numpy()
        for e, o in zip(sample, oracles):
            act = int(a_h[e])
            if rep == "wide":
                act = O.actionmap_unravel(act, shape[0], shape[1], env.n_tiles)
            r, _, _ = o.step(act)
            assert st_h[e].tolist() == O.stats_vector(problem, o.stats), (t, e)
            assert np.array_equal(maps_h[e], o.grid), (t, e)
            assert r_h[e] == pytest.approx(float(r), rel=1e-6, abs=1e-7), (t, e)
    assert torch.equal(env.compute_stats(env.maps), env.stats)    # incremental == recomputed from scratch
    assert torch.equal(env.iteration, torch.full_like(env.iteration, 48))
    env.check_status()


def test_episode_end_and_auto_reset():
    n = 512
    env = _mk("binary", "narrow", (16, 16), n, auto_reset=True, max_board_scans=0.05)   # 256*0.05+1 = 13.8
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(1)
    for t in range(1, 15):
        a = torch.randint(0, 2, (n,), generator=g, device=env.device, dtype=torch.int32)
        _, done = env.step(a)
        if t <= 13:
            assert not bool(done.any()), t
            assert int(env.iteration[0]) == t
        else:
            assert bool(done.all())
            assert int(env.iteration.max()) == 0          # auto-reset happened
            assert torch.equal(env.compute_stats(env.maps), env.stats)


def test_random_reset_distribution_and_determinism():
    env1 = _mk("zelda", "turtle", (7, 11), 4096, seed=11)
    env2 = _mk("zelda", "turtle", (7, 11), 4096, seed=11)
    env1.reset()
    env2.reset()
    assert torch.equal(env1.maps, env2.maps) and torch.equal(env1.pos, env2.pos)
    m = env1.maps
    assert int(m.min()) >= 0 and int(m.max()) <= 7
    assert int(env1.pos[:, 0].max()) <= 6 and int(env1.pos[:, 1].max()) <= 10 and int(env1.pos.min()) >= 0
    env1.reset()
    assert not torch.equal(env1.maps, env2.maps)           # new epoch -> new maps
    env3 = _mk("zelda", "turtle", (7, 11), 4096, seed=11, env_offset=4096)
    env3.reset()
    assert not torch.equal(env3.maps, env2.maps)           # different shard -> different stream
    # fixed init probs: empirical tile frequencies match zelda_prob.py:26
    import control_pcgrl_b200 as P
    env4 = P.BatchedPcgrlEnv(P.make_config("zelda", "narrow"), 8192, random_init_probs=False)
    env4.reset()
    freq = torch.bincount(env4.maps.flatten().long(), minlength=8).double() / env4.maps.numel()
    want = torch.tensor([0.58, 0.3, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02], dtype=torch.float64)
    assert float((freq.cpu() - want).abs().max()) < 5e-3


def test_host_step_and_facade():
    import control_pcgrl_b200 as P
    tr = Trace("binary_narrow")
    d = tr.envs[0]
    # host-buffer path (what bench.py times as e2e)
    env = _mk("binary", "narrow", (16, 16), 1, weights=tr.weights)
    env.reset(grids=d["grid0"][None])
    for t in range(60):
        r, dn, st = env.step_host(np.array([d["actions"][t]], dtype=np.int32))
        assert st[0].tolist() == [int(v) for v in d["stats"][t]]
        assert r[0] == pytest.approx(float(d["rewards"][t]), rel=1e-6, abs=1e-7)
    # single-env façade with the reference's wrapper stack
    cfg = P.make_config("binary", "narrow", weights=tr.weights)
    fenv = P.make_env(cfg)
    fenv.unwrapped.set_map(d["grid0"])
    ob, info = fenv.reset()
    assert ob.shape == (32, 32, 3)
    assert fenv.unwrapped._rep_stats == {"regions": int(d["stats0"][0]), "path-length": int(d["stats0"][1])}
    for t in range(100):
        ob, r, done, trunc, info = fenv.step(int(d["actions"][t]))
        assert r == pytest.approx(float(d["rewards"][t]), rel=1e-6, abs=1e-7)
        assert info["iterations"] == t + 1 and info["changes"] == int(d["changes"][t])
        if t in d["obs_step"]:
            np.testing.assert_array_equal(ob, d["obs"][list(d["obs_step"]).index(t)])
    assert fenv.action_space.n == 2


@pytest.mark.parametrize("problem,rep,shape,controls", [("binary", "narrow", (16, 16), None),
                                                        ("binary", "wide", (16, 16), ["regions", "path-length"]),
                                                        ("zelda", "turtle", (7, 11), None)])
def test_pipelined_host_step_equals_device_step(problem, rep, shape, controls, monkeypatch):
    """pcgrl_step_host cuts big shards into chunks pipelined over helper streams; every chunking must give
    exactly what one whole-shard pcgrl_step gives (ragged last chunk, per-env targets, auto-reset ordering)."""
    n = 70_001
    kw = dict(obs_window=shape) if rep == "wide" else {}
    a = _mk(problem, rep, shape, n, controls=controls, seed=3, auto_reset=True, max_board_scans=0.05, **kw)
    b = _mk(problem, rep, shape, n, controls=controls, seed=3, auto_reset=True, max_board_scans=0.05, **kw)
    if controls:
        g = torch.Generator(device=a.device).manual_seed(1)
        a.sample_uniform_targets(generator=g)
        b.targets.copy_(a.targets)
    a.reset()
    b.reset()
    assert torch.equal(a.grids, b.grids)
    n_act = {"narrow": a.n_tiles, "turtle": 4 + a.n_tiles, "wide": shape[0] * shape[1] * a.n_tiles}[rep]
    rng = np.random.default_rng(0)
    pinned = a.host_action_buffer(None)
    for t, chunks in enumerate(["1", "2", "5", "7", "", "64", "3", "4"] * 3):
        if chunks:
            monkeypatch.setenv("PCGRL_HOST_CHUNKS", chunks)
        else:
            monkeypatch.delenv("PCGRL_HOST_CHUNKS", raising=False)
        act = rng.integers(0, n_act, size=n).astype(np.int32)
        if t % 2:
            pinned.numpy()[...] = act
            r, d, s = a.step_host(pinned)
        else:
            r, d, s = a.step_host(act)
        rb, db = b.step(torch.from_numpy(act).to(b.device))
        # b.step's auto-reset already ran; its reward/done still hold the finishing step's outputs
        np.testing.assert_array_equal(r, rb.cpu().numpy())
        np.testing.assert_array_equal(d, db.cpu().numpy())
        assert torch.equal(a.grids, b.grids) and torch.equal(a.stats, b.stats) and torch.equal(a.pos, b.pos)
        assert torch.equal(a.iteration, b.iteration) and torch.equal(a.changes, b.changes)
    a.check_status()


@pytest.mark.parametrize("problem,rep,shape,controls", [("binary", "narrow", (16, 16), None),
                                                        ("binary", "wide", (16, 16), ["regions", "path-length"]),
                                                        ("zelda", "turtle", (7, 11), None),
                                                        ("sokoban", "narrow", (5, 5), None)])
def test_compact_host_io_equals_int32_outputs(problem, rep, shape, controls, monkeypatch):
    """ABI 5 compact host I/O: uint8 / uint16 actions in, ONE packed record array out (reward f32 | stats u8 or i16
    | done | changed).  Every field must equal the int32 ABI's outputs on the same env, for every chunking."""
    n = 33_333 if problem != "sokoban" else 4_099
    kw = dict(obs_window=shape) if rep == "wide" else {}
    import control_pcgrl_b200 as P
    cfg = P.make_config(problem, rep, map_shape=shape, controls=controls, max_board_scans=0.1, **kw)
    a = P.BatchedPcgrlEnv(cfg, n, seed=7, auto_reset=True, compact_host_io=True)
    b = P.BatchedPcgrlEnv(cfg, n, seed=7, auto_reset=True)
    want_act = {"narrow": np.uint8, "turtle": np.uint8, "wide": np.uint16}[rep]
    assert a.action_shape_dtype()[1] == want_act and b.action_shape_dtype()[1] == np.int32
    want_sb = {"binary": 1, "zelda": 2, "sokoban": 2}[problem]
    assert a.record_dtype()["stats"].base.itemsize == want_sb
    assert a.record_stride == (4 + a.K * want_sb + 2 + 3) // 4 * 4
    if controls:
        g = torch.Generator(device=a.device).manual_seed(1)
        a.sample_uniform_targets(generator=g)
        b.targets.copy_(a.targets)
    a.reset()
    b.reset()
    # resets refresh the stats part of the records
    rec0 = a.records.cpu().numpy().view(a.record_dtype()).reshape(n)
    np.testing.assert_array_equal(rec0["stats"].astype(np.int32), b.stats.cpu().numpy())
    n_act = {"narrow": a.n_tiles, "turtle": 4 + a.n_tiles, "wide": shape[0] * shape[1] * a.n_tiles}[rep]
    rng = np.random.default_rng(0)
    h2d, d2h = a.host_io_bytes()
    assert h2d == n * np.dtype(want_act).itemsize and d2h == n * a.record_stride
    for t, chunks in enumerate(["1", "3", "", "8"] * 4):
        if chunks:
            monkeypatch.setenv("PCGRL_HOST_CHUNKS", chunks)
        else:
            monkeypatch.delenv("PCGRL_HOST_CHUNKS", raising=False)
        act = rng.integers(0, n_act, size=n)
        r, d, s = a.step_host(act.astype(want_act))
        changed_a = a._host_io().views[3].copy()
        r, d, s = r.copy(), d.copy(), s.copy()
        rb, db, sb = b.step_host(act.astype(np.int32))
        np.testing.assert_array_equal(r, rb)
        np.testing.assert_array_equal(d, db)
        # both paths download before the auto-reset launches
        np.testing.assert_array_equal(s.astype(np.int32), sb)
        np.testing.assert_array_equal(changed_a, b.changed.cpu().numpy())
        assert torch.equal(a.grids, b.grids) and torch.equal(a.stats, b.stats)
        # the device-side int32 views stay valid next to the records
        assert torch.equal(a.reward, b.reward) and torch.equal(a.done, b.done)
    a.check_status()
    b.check_status()
    # a device-resident step also keeps the records current (pcgrl_step writes them)
    act = torch.from_numpy(rng.integers(0, n_act, size=n).astype(np.int32))
    shape_a, _, tdt = a._action_layout()
    ra, da = a.step(act.to(tdt).to(a.device))
    rb, db = b.step(act.to(b.device))
    rec = a.records.cpu().numpy().view(a.record_dtype()).reshape(n)
    live = ~db.cpu().numpy().astype(bool)          # finished envs were auto-reset: their stats moved on
    np.testing.assert_array_equal(rec["reward"], rb.cpu().numpy())
    np.testing.assert_array_equal(rec["done"], db.cpu().numpy())
    np.testing.assert_array_equal(rec["stats"].astype(np.int32)[live], b.stats.cpu().numpy()[live])


def test_env_on_non_current_device_and_status_bits():
    """The C ABI launches on the thread's current device: BatchedPcgrlEnv must switch to its own device for every
    call (ADVICE r1), and check_status must name the condition behind each status bit."""
    import control_pcgrl_b200 as P
    env = P.BatchedPcgrlEnv(P.make_config("binary", "narrow"), 256, device="cuda:0")
    env.reset()
    for bit, exc in ((1, ValueError), (2, IndexError), (4, RuntimeError), (8, RuntimeError), (16, OverflowError)):
        env.status.fill_(bit)
        with pytest.raises(exc):
            env.check_status()
        assert int(env.status.item()) == 0
    env.status.fill_(1 | 4)
    with pytest.raises(RuntimeError, match="workspace"):
        env.check_status()
    bad = torch.full((256,), 7, dtype=torch.int32, device=env.device)
    env.step(bad)
    with pytest.raises(ValueError, match="action"):
        env.check_status()
    if torch.cuda.device_count() < 2:
        return
    torch.cuda.set_device(0)
    e1 = P.BatchedPcgrlEnv(P.make_config("binary", "narrow"), 4096, device="cuda:1", seed=3)
    e0 = P.BatchedPcgrlEnv(P.make_config("binary", "narrow"), 4096, device="cuda:0", seed=3)
    e1.reset()
    e0.reset()
    act = torch.randint(0, 2, (4096,), dtype=torch.int32)
    for _ in range(5):
        r1, _ = e1.step(act.to("cuda:1"))
        r0, _ = e0.step(act.to("cuda:0"))
    assert torch.equal(e1.grids.cpu(), e0.grids.cpu()) and torch.equal(e1.stats.cpu(), e0.stats.cpu())
    assert torch.equal(r1.cpu(), r0.cpu())
    assert torch.equal(e1.observe(dtype=torch.uint8).cpu(), e0.observe(dtype=torch.uint8).cpu())


def test_static_tiles_random_reset_and_frozen_cells():
    """StaticTileRepresentation (envs/reps/wrappers.py:234-376) at scale: the random-reset generator
    (static_prob / n_static_walls) and the invariant that a frozen cell never changes while its attempted
    edits are still counted as changes."""
    n = 16384
    env = _mk("binary", "narrow", (16, 16), n, seed=5, static_tile_wrapper=True, static_prob=0.6, n_static_walls=3)
    env.reset()
    sm = env.static_tiles.clone()
    g0 = env.maps.clone()
    frac = sm.float().mean(dim=(1, 2))                       # per-episode probability U(0,1) * 0.6, plus walls
    assert 0.25 < float(frac.mean()) < 0.40 and float(frac.max()) < 0.75
    assert float(frac.std()) > 0.1                           # the probability is drawn per episode
    assert torch.equal(env.compute_stats(env.maps), env.stats)
    # walls: frozen cells at wall_pos - 1, wall tiles (solid) one cell further along both axes
    env2 = _mk("binary", "narrow", (16, 16), n, seed=5, static_tile_wrapper=True, static_prob=0.0, n_static_walls=1)
    env2.reset()
    sm2, g2 = env2.static_tiles, env2.maps
    cnt = sm2.sum(dim=(1, 2))
    assert int(cnt.min()) >= 1 and int(cnt.max()) <= 14      # integers(1, 15) cells in one straight segment
    rows, cols = sm2.any(dim=2).sum(dim=1), sm2.any(dim=1).sum(dim=1)
    assert bool(((rows == 1) | (cols == 1)).all())
    shifted = torch.zeros_like(sm2)
    shifted[:, 1:, 1:] = sm2[:, :-1, :-1]
    assert bool((g2[shifted.bool()] == 1).all())
    # rollout: frozen cells keep their tile, changes still count attempts
    gen = torch.Generator(device=env.device).manual_seed(1)
    attempts = torch.zeros(n, dtype=torch.int32, device=env.device)
    for t in range(300):
        a = torch.randint(0, 2, (n,), generator=gen, device=env.device, dtype=torch.int32)
        pos = env.pos.clone()
        cur = env.maps[torch.arange(n, device=env.device), pos[:, 0].long(), pos[:, 1].long()]
        attempts += (cur.int() != a).int()
        prev_stats = env.stats.clone()
        reward, _ = env.step(a)
        froz = sm[torch.arange(n, device=env.device), pos[:, 0].long(), pos[:, 1].long()].bool()
        undone = froz & (cur.int() != a)
        assert torch.equal(env.stats[undone], prev_stats[undone]) and bool((reward[undone] == 0).all())
    assert torch.equal(env.changes, attempts)
    assert torch.equal(env.maps[sm.bool()], g0[sm.bool()])
    assert not torch.equal(env.maps, g0)
    assert torch.equal(env.compute_stats(env.maps), env.stats)
    obs = env.observe(dtype=torch.uint8)
    assert obs.shape == (n, 32, 32, 4)
    env.check_status()


@pytest.mark.parametrize("problem,shape,aw", [("binary", (16, 16), (2, 2)), ("binary", (16, 16), (16, 1)),
                                              ("binary", (16, 16), (16, 16)), ("zelda", (7, 11), (3, 4))])
def test_action_patch_rollout_vs_oracle(problem, shape, aw):
    """MultiActionRepresentation (cfg.act_window) on random rollouts against the oracle, incl. the squeegee and
    whole-map patches of configs/experiment/{action_patch,squeegee}.yaml."""
    from oracle import pcgrl_oracle as O
    n, steps = 24, 40
    rng = np.random.default_rng(7)
    nt = len(O.TILES[problem])
    grids = rng.integers(0, nt, size=(n, *shape)).astype(np.int8)
    env = _mk(problem, "narrow", shape, n, act_window=aw)
    env.reset(grids=grids)
    oracles = []
    for e in range(n):
        o = O.OracleEnv(problem, "narrow", shape, weights=dict(env.metric_weights), act_window=aw)
        o.reset(grids[e])
        oracles.append(o)
    for t in range(steps):
        a = rng.integers(0, nt, size=(n, int(np.prod(aw)))).astype(np.int32)
        if t % 3 == 2:
            for e, o in enumerate(oracles):   # no-op patches
                tl = [o.pos[i] - (aw[i] - 1) // 2 for i in range(2)]
                a[e] = o.grid[tl[0]:tl[0] + aw[0], tl[1]:tl[1] + aw[1]].reshape(-1)
        reward, done = env.step(torch.from_numpy(a).to(env.device))
        reward, stats, maps, pos = reward.cpu().numpy(), env.stats.cpu().numpy(), env.maps.cpu().numpy(), env.pos.cpu().numpy()
        for e, o in enumerate(oracles):
            r, d, _ = o.step(a[e])
            assert stats[e].tolist() == O.stats_vector(problem, o.stats), (t, e)
            assert np.array_equal(maps[e], o.grid) and pos[e, :2].tolist() == o.pos, (t, e)
            assert reward[e] == pytest.approx(r, rel=1e-6, abs=1e-7)
    assert env.changes.cpu().numpy().tolist() == [o.changes for o in oracles]
    env.check_status()


@pytest.mark.parametrize("problem,rep,shape,obs", [("binary", "narrow", (16, 16), (32, 32)),
                                                   ("zelda", "turtle", (7, 11), (22, 22)),
                                                   ("minecraft_3D_maze", "narrow", (6, 7, 8), (12, 14, 16)),
                                                   ("binary", "wide", (16, 16), (16, 16))])
def test_tile_code_observation_is_the_argmax_of_the_onehot(problem, rep, shape, obs):
    """observe(onehot=False) = Cropped's own output: the channel index of the one-hot record of every pixel."""
    for n in (5, 64):
        env = _mk(problem, rep, shape, n, obs_window=obs, seed=n, action_kind="wide_flat" if rep == "wide" else None)
        env.reset()
        if rep in ("narrow", "turtle"):
            for i, d in enumerate(shape):
                env.pos[:, i] = torch.randint(0, d, (n,), device=env.device, dtype=torch.int32)
        onehot = env.observe(dtype=torch.uint8)
        raw = env.observe(onehot=False)
        assert raw.shape == (*onehot.shape[:-1], 1) and raw.dtype == torch.uint8
        assert torch.equal(raw[..., 0].long(), onehot.argmax(dim=-1))
        assert int(onehot.sum()) == raw[..., 0].numel()


@pytest.mark.parametrize("shape,obs", [((16, 16), (32, 32)), ((10, 16), (20, 32)), ((5, 12), (10, 32)), ((16, 9), (32, 32))])
def test_row_per_thread_observation_writer(shape, obs):
    """Two-tile crops whose window is exactly 32 wide take the 32-pixels-per-thread path of the staged writer (a whole
    window row from two funnel shifts and eight table lookups): uint8 one-hot and tile codes must equal the float
    writer's output (which shares none of that code), for positions all over the map, ragged last trips included."""
    for n in (5, 333, 4099):
        env = _mk("binary", "narrow", shape, n, obs_window=obs, seed=n)
        env.reset()
        for i, d in enumerate(shape):
            env.pos[:, i] = torch.randint(0, d, (n,), device=env.device, dtype=torch.int32)
        env.pos[0, 0], env.pos[0, 1] = 0, 0
        env.pos[1, 0], env.pos[1, 1] = shape[0] - 1, shape[1] - 1
        want = env.observe(dtype=torch.float32)
        u8 = env.observe(dtype=torch.uint8)
        codes = env.observe(onehot=False)
        assert torch.equal(u8.float(), want)
        assert torch.equal(codes[..., 0].long(), want.argmax(dim=-1))


def test_zelda_u8_observation_rows_per_thread():
    """zelda's 22-wide window takes 11 pixels (half a window row) per thread in the staged u8 writer; it must equal the
    float writer, with positions all over the map."""
    for n in (3, 1000):
        env = _mk("zelda", "turtle", (7, 11), n, obs_window=(22, 22), seed=n)
        env.reset()
        for i, d in enumerate((7, 11)):
            env.pos[:, i] = torch.randint(0, d, (n,), device=env.device, dtype=torch.int32)
        want = env.observe(dtype=torch.float32)
        assert torch.equal(env.observe(dtype=torch.uint8).float(), want)
        assert torch.equal(env.observe(onehot=False)[..., 0].long(), want.argmax(dim=-1))


def test_maze3d_u8_observation_rows_per_thread():
    """The 3D maze's 14-wide last window axis: 7 pixels per thread in the staged u8 writer against the float writer."""
    for n in (3, 700):
        env = _mk("minecraft_3D_maze", "narrow", (14, 14, 14), n, obs_window=(14, 14, 14), seed=n)
        env.reset()
        for i in range(3):
            env.pos[:, i] = torch.randint(0, 14, (n,), device=env.device, dtype=torch.int32)
        want = env.observe(dtype=torch.float32)
        assert torch.equal(env.observe(dtype=torch.uint8).float(), want)
        assert torch.equal(env.observe(onehot=False)[..., 0].long(), want.argmax(dim=-1))
