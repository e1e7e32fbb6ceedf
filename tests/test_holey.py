"""Holey problems (SURVEY 8f rank 2): binary_holey -- stats on the bordered map with an entrance and an exit.

The reference's holey *env classes* cannot be constructed at this commit (pcgrl_holey_env.py:32-33 passes
(prob, rep) to a constructor that takes (cfg, prob, rep); BinaryHoleyProblem.__init__ calls BinaryProblem.__init__
without the cfg it requires), so parity is pinned on what still runs verbatim: BinaryHoleyProblem.get_stats,
_valid_holes and get_border_idxs, through tests/golden/stats_binary_holey.npz (oracle/gen_golden.py).
"""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "stats_binary_holey.npz")


def _groups():
    z = np.load(GOLDEN)
    i = 0
    while f"grids_{i}" in z:
        yield i, z[f"grids_{i}"], z[f"holes_{i}"], z[f"stats_{i}"], z
        i += 1


# ------------------------------------------------------------------------------------------ CPU: oracle pinned
def test_oracle_matches_reference_get_stats():
    from oracle import pcgrl_oracle as O
    total = 0
    for _, grids, holes, stats, _ in _groups():
        for g, h, s in zip(grids, holes, stats):
            assert O.stats_vector("binary_holey", O.binary_holey_stats(g, h)) == s.tolist()
            total += 1
    assert total >= 700


def test_oracle_hole_rules_match_reference():
    from oracle import pcgrl_oracle as O
    for gi, grids, _, _, z in _groups():
        h, w = grids.shape[1:]
        border = O.holey_border_idxs(h, w)
        assert np.array_equal(border, z[f"border_{gi}"])
        for (a, b), v in zip(z[f"valid_pairs_{gi}"], z[f"valid_{gi}"]):
            assert O.valid_holes(border[a], border[b], h, w) == bool(v)


def test_spec_constants_match_oracle():
    import control_pcgrl_b200.problems as PR
    from oracle import pcgrl_oracle as O
    for shape in [(16, 16), (10, 14)]:
        s = PR.get_spec("binary_holey", shape)
        c = O.problem_constants("binary_holey", shape)
        assert s.stat_names == O.STAT_NAMES["binary_holey"]
        assert {k: float(v) for k, v in s.static_trgs.items()} == {k: float(v) for k, v in c["static_trgs"].items()}
        assert {k: tuple(map(float, v)) for k, v in s.cond_bounds.items()} == \
            {k: tuple(map(float, v)) for k, v in c["cond_bounds"].items()}
        assert s.reward_weights == c["default_weights"]


# ------------------------------------------------------------------------------------------ GPU
def _mk(shape, n, **kw):
    import control_pcgrl_b200 as P
    cfg = P.make_config("binary_holey", kw.pop("rep", "narrow"), map_shape=shape,
                        weights={"regions": 1, "path-length": 2, "connected-path-length": 3},
                        **{k: kw.pop(k) for k in list(kw) if k in ("fixed_holes", "max_board_scans", "change_percentage")})
    return P.BatchedPcgrlEnv(cfg, n, **kw)


@pytest.mark.gpu
def test_stats_kernel_matches_reference_fixture():
    total = 0
    for _, grids, holes, stats, _ in _groups():
        env = _mk(grids.shape[1:], 1)
        got = env.compute_stats(grids, holes=holes).cpu().numpy()
        bad = np.flatnonzero((got != stats).any(axis=1))
        assert bad.size == 0, (grids.shape, bad[:5], got[bad[:5]], stats[bad[:5]], holes[bad[:5]])
        total += len(grids)
    assert total >= 700


@pytest.mark.gpu
@pytest.mark.parametrize("rep,shape", [("narrow", (16, 16)), ("turtle", (9, 12)), ("wide", (16, 16))])
def test_rollout_vs_oracle(rep, shape):
    import torch
    from oracle import pcgrl_oracle as O
    rng = np.random.default_rng(5)
    n, steps = 24, 120
    h, w = shape
    border = O.holey_border_idxs(h, w)
    grids = (rng.random((n, h, w)) < 0.45).astype(np.int8)
    holes = np.array([np.concatenate([border[k] for k in rng.choice(len(border), 2, replace=False)]) for _ in range(n)],
                     dtype=np.int32)
    pos0 = np.stack([rng.integers(0, h, n), rng.integers(0, w, n)], axis=1)
    env = _mk(shape, n, rep=rep, action_kind="wide_coords" if rep == "wide" else None)
    env.reset(grids=grids, holes=holes, pos=pos0 if rep == "turtle" else None)
    weights = {"regions": 1, "path-length": 2, "connected-path-length": 3}
    oracles = []
    for e in range(n):
        o = O.OracleEnv("binary_holey", rep, shape, weights=weights)
        o.reset(grids[e], pos=pos0[e] if rep == "turtle" else None, holes=holes[e])
        oracles.append(o)
    assert env.stats.cpu().numpy().tolist() == [O.stats_vector("binary_holey", o.stats) for o in oracles]
    for t in range(steps):
        if rep == "narrow":
            a = rng.integers(0, 2, n).astype(np.int32)
        elif rep == "turtle":
            a = rng.integers(0, 6, n).astype(np.int32)
        else:
            a = np.stack([rng.integers(0, h, n), rng.integers(0, w, n), rng.integers(0, 2, n)], axis=1).astype(np.int32)
        reward, done = env.step(torch.from_numpy(a).to(env.device))
        reward, done = reward.cpu().numpy(), done.cpu().numpy()
        stats, maps = env.stats.cpu().numpy(), env.maps.cpu().numpy()
        for e, o in enumerate(oracles):
            r, d, _ = o.step(a[e].tolist() if rep == "wide" else int(a[e]))
            assert stats[e].tolist() == O.stats_vector("binary_holey", o.stats), (t, e)
            assert np.array_equal(maps[e], o.grid), (t, e)
            assert bool(done[e]) == d and abs(float(reward[e]) - r) <= 1e-6 * max(1.0, abs(r)), (t, e, reward[e], r)
    env.check_status()


@pytest.mark.gpu
def test_random_and_fixed_holes_on_reset():
    from oracle import pcgrl_oracle as O
    h, w, n = 16, 16, 4096
    env = _mk((h, w), n, seed=3)
    env.reset()
    holes = env.holes.cpu().numpy()
    border = {tuple(b) for b in O.holey_border_idxs(h, w).tolist()}
    ent, ext = holes[:, :2], holes[:, 2:]
    assert all(tuple(e) in border for e in ent.tolist()) and all(tuple(e) in border for e in ext.tolist())
    assert (ent != ext).any(axis=1).all()
    # the reference's rule: the exit is a candidate that _valid_holes accepts (or, rarely, the fallback)
    ok = np.array([O.valid_holes(e, x, h, w) for e, x in zip(ent, ext)])
    assert ok.mean() > 0.98
    assert len({tuple(r) for r in holes.tolist()}) > 1000            # spread over the border
    # stats of the drawn maps + holes agree with the oracle
    maps = env.maps.cpu().numpy()
    st = env.stats.cpu().numpy()
    for e in range(0, n, 97):
        assert st[e].tolist() == O.stats_vector("binary_holey", O.binary_holey_stats(maps[e], holes[e]))
    # determinism and a new draw per episode
    env2 = _mk((h, w), n, seed=3)
    env2.reset()
    assert np.array_equal(env2.holes.cpu().numpy(), holes)
    env.reset()
    assert not np.array_equal(env.holes.cpu().numpy(), holes)
    # fixed_holes: entrance (1, 0), exit (W, H + 1)   (holey_prob.py:47-49)
    envf = _mk((h, w), 64, fixed_holes=True)
    envf.reset()
    assert (envf.holes.cpu().numpy() == np.array([1, 0, w, h + 1])).all()


@pytest.mark.gpu
@pytest.mark.parametrize("rep,shape,window", [("narrow", (16, 16), (32, 32)), ("turtle", (9, 12), (18, 24)),
                                              ("wide", (10, 10), (10, 10))])
def test_holey_observation_matches_oracle(rep, shape, window):
    """HoleyRepresentation.get_observation (envs/reps/wrappers.py:153-174): the bordered map with the two holes,
    positions + 1, through the usual Cropped / OneHot stack whose window is then two cells larger."""
    import torch
    from oracle import pcgrl_oracle as O
    import control_pcgrl_b200 as P
    rng = np.random.default_rng(3)
    n = 37
    h, w = shape
    border = O.holey_border_idxs(h, w)
    grids = (rng.random((n, h, w)) < 0.5).astype(np.int8)
    holes = np.array([np.concatenate([border[k] for k in rng.choice(len(border), 2, replace=False)]) for _ in range(n)],
                     dtype=np.int32)
    cfg = P.make_config("binary_holey", rep, map_shape=shape, obs_window=window)
    env = P.BatchedPcgrlEnv(cfg, n, action_kind="wide_coords" if rep == "wide" else None)
    pos = np.stack([rng.integers(0, h, n), rng.integers(0, w, n)], axis=1)
    env.reset(grids=grids, holes=holes, pos=pos if rep == "turtle" else None)
    if rep == "narrow":
        env.pos[:, :2] = torch.from_numpy(pos).to(env.device, torch.int32)
    obs = env.observe(dtype=torch.float64).cpu().numpy()
    codes = env.observe(onehot=False).cpu().numpy()[..., 0]
    # the staged writer (default) and the pixel-per-thread writer agree, every dtype: an output view one element past
    # a 16-byte boundary takes the pixel writer
    for dt in (torch.uint8, torch.float32, torch.float64):
        a = env.observe(dtype=dt)
        view = torch.empty(a.numel() + 1, dtype=dt, device=env.device)[1:].view(a.shape)
        assert view.data_ptr() % 16 != 0
        assert torch.equal(env.observe(out=view), a), (rep, dt)
    ow = tuple(d + 2 for d in (window if rep != "wide" else shape))
    assert obs.shape == (n, *ow, 3 if rep != "wide" else 2)
    for e in range(n):
        b = O.bordered_with_holes(grids[e], holes[e])
        if rep == "wide":
            want = O.full_onehot(b, 2)
        else:
            want = O.cropped_onehot(b, [int(pos[e, 0]) + 1, int(pos[e, 1]) + 1], ow, 2)
        assert np.array_equal(obs[e], want), (rep, e)
        assert np.array_equal(codes[e], want.argmax(-1)), (rep, e)


@pytest.mark.gpu
def test_single_env_facade():
    """make("binary_holey-narrow-v0"): bordered observation with the holes, pos + 1, queued holes, get_stats on
    the bordered string map (what PcgrlEnv.step hands the problem, pcgrl_env.py:323)."""
    import control_pcgrl_b200 as P
    from oracle import pcgrl_oracle as O
    env = P.make("binary_holey-narrow-v0")
    assert env.observation_space["map"].shape == (34, 34)
    env.unwrapped._prob.queue_holes([((0, 3), (17, 9))])
    grid = (np.random.default_rng(1).random((16, 16)) < 0.4).astype(np.int8)
    env.set_map(grid)
    obs, _ = env.reset()
    assert obs["map"].shape == (18, 18) and obs["map"][0, 3] == 0 and obs["map"][17, 9] == 0
    assert obs["map"][0, 4] == 1 and obs["pos"].tolist() == [1, 1]
    assert np.array_equal(obs["map"][1:-1, 1:-1], grid)
    want = O.binary_holey_stats(grid, [0, 3, 17, 9])
    assert dict(env.unwrapped._rep_stats) == want
    tiles = env.unwrapped._prob.get_tile_types()
    smap = [[tiles[v] for v in row] for row in obs["map"]]
    assert dict(env.unwrapped._prob.get_stats(smap)) == want
    obs, _, done, _, info = env.step(1 - int(grid[0, 0]))
    grid[0, 0] = 1 - grid[0, 0]
    assert info["regions"] == O.binary_holey_stats(grid, [0, 3, 17, 9])["regions"]
    assert obs["pos"].tolist() == [1, 1]      # narrow: cell 0 is edited twice (narrow_rep.py:98-100)


@pytest.mark.gpu
def test_full_size_incremental_stats_equal_recomputed():
    """65 536 envs, random holes: after a rollout the incrementally maintained stats equal get_stats recomputed from
    scratch on the final maps (size-independent property), unchanged envs got exactly 0 reward, and a sample agrees
    with the oracle."""
    import torch
    from oracle import pcgrl_oracle as O
    n = 65536
    env = _mk((16, 16), n, seed=8)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(1)
    for _ in range(30):
        a = torch.randint(0, 2, (n,), generator=g, device=env.device, dtype=torch.int32)
        reward, _ = env.step(a)
        unchanged = env.changed == 0
        assert bool((reward[unchanged] == 0).all())
    again = env.compute_stats(env.maps, holes=env.holes)
    assert torch.equal(again, env.stats)
    maps, holes, stats = env.maps.cpu().numpy(), env.holes.cpu().numpy(), env.stats.cpu().numpy()
    for e in range(0, n, 4099):
        assert stats[e].tolist() == O.stats_vector("binary_holey", O.binary_holey_stats(maps[e], holes[e]))
    env.check_status()


def test_maze3d_holey_oracle_matches_reference_get_stats():
    """minecraft_3D_holey_maze (oracle only so far; the CUDA path is round-2 work): the restatement -- one search
    from the entrance keeping the path lists, connected length / jumps at the exit, and `path-length` = the
    de-stacked longest path of the PREVIOUS call -- against sequences of calls on the reference's problem object
    (tests/golden/stats_maze3d_holey.npz, oracle/gen_golden.py)."""
    from oracle import maze3d_oracle as M
    z = np.load(os.path.join(os.path.dirname(GOLDEN), "stats_maze3d_holey.npz"))
    total, connected, stale = 0, 0, 0
    gi = 0
    while f"maps_{gi}" in z:
        maps, holes, stats, steps = z[f"maps_{gi}"], z[f"holes_{gi}"], z[f"stats_{gi}"], int(z[f"steps_{gi}"])
        prev = 0
        for i in range(len(maps)):
            if i % steps == 0:
                prev = 0                                   # a fresh problem object: path_coords = []
            st, prev = M.maze3d_holey_stats(maps[i], holes[i][0], holes[i][1], prev)
            got = [st[k] for k in ("regions", "path-length", "connected-path-length", "n_jump")]
            assert got == stats[i].tolist(), (gi, i, got, stats[i])
            total += 1
            connected += stats[i][2] > 0
            stale += stats[i][1] > 0
        gi += 1
    assert total >= 290 and connected >= 20 and stale >= 100


# ---------------------------------------------------------------------------------------------------------------
# the 3D holey problems on the GPU (SURVEY 8f rank 2): minecraft_3D_holey_maze, minecraft_3D_dungeon_holey
# ---------------------------------------------------------------------------------------------------------------
import torch  # noqa: E402
from oracle import pcgrl_oracle as O  # noqa: E402


def _holes6(h):
    """fixture holes [n, 2 (entrance, exit), 2 (foot, head), 3 (z, y, x)] -> the kernel's [n, 6] foot tiles"""
    return np.concatenate([h[:, 0, 0, :], h[:, 1, 0, :]], axis=1).astype(np.int32)


def test_maze3d_holey_dungeon_oracle_matches_reference_get_stats():
    from oracle import maze3d_oracle as M
    z = np.load(os.path.join(os.path.dirname(GOLDEN), "stats_maze3d_holey_dungeon.npz"))
    n = 0
    for gi in range(3):
        for b, h, want in zip(z[f"maps_{gi}"], z[f"holes_{gi}"], z[f"stats_{gi}"]):
            st = M.maze3d_holey_dungeon_stats(b, h[0], h[1])
            assert [int(st[k]) for k in O.STAT_NAMES["minecraft_3D_dungeon_holey"]] == want.tolist()
            n += 1
    assert n == 176


@pytest.mark.gpu
def test_maze3d_holey_kernel_matches_reference_fixture():
    """minecraft_3D_holey_maze get_stats on the GPU against 291 sequential calls of the reference's problem object:
    path-length is the de-stacked longest path of the PREVIOUS call (minecraft_3D_holey_maze_prob.py:92-93), so each
    trial's calls are replayed in order, carrying `_next-path-length`."""
    import control_pcgrl_b200 as P
    z = np.load(os.path.join(os.path.dirname(GOLDEN), "stats_maze3d_holey.npz"))
    total = 0
    for gi in range(3):
        maps, holes, stats, steps = z[f"maps_{gi}"], z[f"holes_{gi}"], z[f"stats_{gi}"], int(z[f"steps_{gi}"])
        size = maps.shape[1] - 2
        trials = len(maps) // steps
        env = P.BatchedPcgrlEnv(P.make_config("minecraft_3D_holey_maze", "narrow", map_shape=(size,) * 3), 1)
        prev = np.zeros(trials, dtype=np.int32)
        for s in range(steps):
            sel = np.arange(trials) * steps + s
            got = env.compute_stats(maps[sel][:, 1:-1, 1:-1, 1:-1], holes=_holes6(holes[sel]),
                                    prev_path_length=prev).cpu().numpy()
            bad = np.flatnonzero((got[:, :4] != stats[sel]).any(axis=1))
            assert bad.size == 0, (gi, s, bad[:4], got[bad[:4]], stats[sel][bad[:4]])
            prev = got[:, 4].astype(np.int32)
            total += len(sel)
        env.check_status()
    assert total == 291


@pytest.mark.gpu
def test_maze3d_holey_dungeon_kernel_matches_reference_fixture():
    import control_pcgrl_b200 as P
    z = np.load(os.path.join(os.path.dirname(GOLDEN), "stats_maze3d_holey_dungeon.npz"))
    total = 0
    for gi in range(3):
        maps, holes, stats = z[f"maps_{gi}"], z[f"holes_{gi}"], z[f"stats_{gi}"]
        size = maps.shape[1] - 2
        env = P.BatchedPcgrlEnv(P.make_config("minecraft_3D_dungeon_holey", "narrow", map_shape=(size,) * 3), 1)
        got = env.compute_stats(maps[:, 1:-1, 1:-1, 1:-1], holes=_holes6(holes)).cpu().numpy()
        bad = np.flatnonzero((got != stats).any(axis=1))
        assert bad.size == 0, (gi, bad[:4], got[bad[:4]], stats[bad[:4]])
        total += len(maps)
        env.check_status()
    assert total == 176


@pytest.mark.gpu
@pytest.mark.parametrize("problem,rep,fixed", [("minecraft_3D_holey_maze", "narrow", False),
                                               ("minecraft_3D_holey_maze", "turtle", True),
                                               ("minecraft_3D_dungeon_holey", "narrow", False),
                                               ("minecraft_3D_dungeon_holey", "wide", True)])
def test_holey3d_rollout_matches_oracle(problem, rep, fixed):
    """Random resets (device-drawn holes: distinct border cells, entrance = the first, exit = the first valid one,
    holey_prob_3D.py:72-100; or the fixed pair), then random edits: every env's stats / reward against the oracle
    env, which carries the holey maze's one-call-late path length across steps and resets."""
    import control_pcgrl_b200 as P
    n, steps, size = 24, 30, 7
    cfg = P.make_config(problem, rep, map_shape=(size,) * 3, fixed_holes=fixed, max_board_scans=0.05)
    env = P.BatchedPcgrlEnv(cfg, n, seed=5, action_kind="wide_coords" if rep == "wide" else None, auto_reset=False)
    n_tiles = env.n_tiles
    rng = np.random.default_rng(1)
    probs = [0.5, 0.5] if n_tiles == 2 else [0.5, 0.38, 0.04, 0.04, 0.04]
    grids = rng.choice(n_tiles, size=(n, size, size, size), p=probs).astype(np.int8)
    env.reset(grids=grids)
    holes = env.holes.cpu().numpy()
    # the generated holes are legal: foot tiles on the side faces (not on a vertical edge, not on the top layer),
    # entrance != exit, and the reference's validity rule between them (or its (1, 1, 1) default)
    for hz in holes:
        for f in (hz[:3], hz[3:]):
            if tuple(f) == (1, 1, 1):
                continue
            on_x = f[2] in (0, size + 1) and 1 <= f[1] <= size
            on_y = f[1] in (0, size + 1) and 1 <= f[2] <= size
            assert 1 <= f[0] <= size - 1 and (on_x != on_y), hz
        if fixed:
            assert hz.tolist() == [1, 0, size, 2, size + 1, 1]
        elif tuple(hz[3:]) != (1, 1, 1):
            d = max(abs(hz[0] - hz[3]), abs(hz[0] + 1 - hz[3]), abs(hz[1] - hz[4]), abs(hz[2] - hz[5]))
            assert d > 1, hz
    pos0 = env.pos.cpu().numpy()
    oracles = []
    for e in range(n):
        o = O.OracleEnv(problem, rep, (size,) * 3, weights=dict(env.metric_weights), max_board_scans=0.05)
        o.reset(grids[e], pos=pos0[e], holes=holes[e])
        oracles.append(o)
    st0 = env.stats.cpu().numpy()
    for e, o in enumerate(oracles):
        assert st0[e].tolist() == O.stats_vector(problem, o.stats), (e, st0[e], o.stats)
    n_act = {"narrow": n_tiles, "turtle": 4 + n_tiles}.get(rep)
    for t in range(steps):
        if rep == "wide":
            a = np.concatenate([rng.integers(0, size, size=(n, 3)), rng.integers(0, n_tiles, size=(n, 1))], axis=1).astype(np.int32)
        else:
            a = rng.integers(0, n_act, size=n).astype(np.int32)
        reward, done = env.step(torch.from_numpy(a).to(env.device))
        r_h, st_h, d_h = reward.cpu().numpy(), env.stats.cpu().numpy(), done.cpu().numpy()
        for e, o in enumerate(oracles):
            r, d, _ = o.step(a[e].tolist() if rep == "wide" else int(a[e]))
            assert st_h[e].tolist() == O.stats_vector(problem, o.stats), (t, e, st_h[e], o.stats)
            assert r_h[e] == pytest.approx(float(r), rel=1e-6, abs=1e-6), (t, e)
            assert bool(d_h[e]) == d
    env.check_status()


@pytest.mark.gpu
@pytest.mark.parametrize("problem", ["minecraft_3D_holey_maze", "minecraft_3D_dungeon_holey"])
@pytest.mark.parametrize("rep", ["narrow", "turtle", "wide"])
def test_maze3d_holey_observation(problem, rep):
    """HoleyRepresentation3D.get_observation (envs/reps/wrappers.py:153-160, 182-185): the bordered 3D map with the
    entrance and the exit dug two tiles high, position + 1, through Cropped + OneHotEncoding (window + 2) -- against
    the restatement, with holes drawn on the device."""
    import control_pcgrl_b200 as P
    rng = np.random.default_rng(21)
    n, size, window = 9, 5, (6, 8, 10)
    spec_tiles = len(O.TILES[problem])
    grids = rng.integers(0, spec_tiles, size=(n, size, size, size)).astype(np.int8)
    cfg = P.make_config(problem, rep, map_shape=(size,) * 3, obs_window=window)
    env = P.BatchedPcgrlEnv(cfg, n, action_kind="wide_coords" if rep == "wide" else None, seed=5)
    pos = rng.integers(0, size, size=(n, 3))
    env.reset(grids=grids, pos=pos if rep == "turtle" else None)
    if rep == "narrow":
        env.pos[:, :3] = torch.from_numpy(pos).to(env.device, torch.int32)
    holes = env.holes.cpu().numpy()
    assert len({tuple(h) for h in holes.tolist()}) > 1          # drawn per env
    obs = env.observe(dtype=torch.float64).cpu().numpy()
    for dt in (torch.uint8, torch.float32):
        assert np.array_equal(env.observe(dtype=dt).cpu().numpy().astype(np.float64), obs)
    codes = env.observe(onehot=False).cpu().numpy()[..., 0]
    ow = tuple(d + 2 for d in (window if rep != "wide" else (size,) * 3))
    assert obs.shape == (n, *ow, spec_tiles + (1 if rep != "wide" else 0))
    dug = 0
    for e in range(n):
        b, ent, ext = O.bordered_with_holes_3d(grids[e], holes[e])
        # the interior of the bordered map is rewritten from the map at every update (representation.py:162-164), so
        # the reference's default exit (1, 1, 1) -- an interior cell -- does not stay dug
        b[1:-1, 1:-1, 1:-1] = grids[e]
        if rep == "wide":
            want = O.full_onehot(b, spec_tiles)
        else:
            want = O.cropped_onehot(b, [int(v) + 1 for v in pos[e]], ow, spec_tiles)
        assert np.array_equal(obs[e], want), (problem, rep, e)
        assert np.array_equal(codes[e], want.argmax(-1)), (problem, rep, e)
        dug += int((b == 0).sum() - (grids[e] == 0).sum())
    assert dug >= 3 * n          # entrance and exit really are in the observed border
