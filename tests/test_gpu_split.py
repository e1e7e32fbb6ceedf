"""GPU: the three equivalent step paths of the bit-board problems must agree bit for bit.

  fused  k_step_bitboard (one launch: update, searches, reward) -- pinned on the reference fixtures elsewhere
  split  k_split_act / k_split_stats / k_split_out (global work list, from-scratch searches with full warps)
  inc    the same with the incremental binary search from the per-env cache (BinaryIncMachine)
  incfused  k_step_inc: update, incremental search and reward in one launch, every warp on its own env slice

PCGRL_STEP_PATH selects the path per pcgrl_step call.  Besides path-vs-path equality, every few steps the stats of
EVERY env are recomputed from scratch from the current grids (pcgrl_stats), which is what pins the incremental
machine: any drift of its cache would show up as a stat that a fresh computation does not give.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _envs(problem, rep, shape, n, paths, **kw):
    import control_pcgrl_b200 as P
    cfg_kw = {k: v for k, v in kw.items() if k in ("controls", "obs_window", "max_board_scans", "change_percentage",
                                                   "act_window", "static_tile_wrapper", "static_prob", "n_static_walls")}
    cfg = P.make_config(problem, rep, map_shape=shape, **cfg_kw)
    return [P.BatchedPcgrlEnv(cfg, n, seed=11, auto_reset=True, split_step=(p != "fused")) for p in paths]


def _n_act(env, rep, shape):
    return {"narrow": env.n_tiles, "turtle": 4 + env.n_tiles, "wide": shape[0] * shape[1] * env.n_tiles}[rep]


CASES = [
    ("binary", "narrow", (16, 16), None),
    ("binary", "turtle", (16, 16), None),
    ("binary", "wide", (16, 16), ["regions", "path-length"]),
    ("binary", "narrow", (10, 10), None),      # generic staging path (rows narrower than 16)
    ("binary", "narrow", (7, 5), None),        # 4-word boards
    ("binary", "turtle", (3, 4), None),        # 2-word boards
    ("binary", "narrow", (2, 16), None),       # 1-word boards
    ("binary", "narrow", (20, 24), None),      # one row per word: split path, no cache
    ("zelda", "turtle", (7, 11), None),
    ("zelda", "narrow", (7, 11), None),
    ("binary_holey", "narrow", (16, 16), None),
]


@pytest.mark.parametrize("problem,rep,shape,controls", CASES)
def test_step_paths_agree_and_match_fresh_stats(problem, rep, shape, controls, monkeypatch):
    n = 12_345
    kw = dict(controls=controls, max_board_scans=0.6)
    if rep == "wide":
        kw["obs_window"] = shape
    paths = ["fused", "split", "inc", "incfused", "lg"]
    envs = _envs(problem, rep, shape, n, paths, **kw)
    has_cache = envs[2].cache is not None
    assert has_cache == (problem == "binary" and max(shape) <= 16)
    assert envs[0].worklist is None and envs[1].worklist is not None
    if controls:
        g = torch.Generator(device=envs[0].device).manual_seed(1)
        envs[0].sample_uniform_targets(generator=g)
        for e in envs[1:]:
            e.targets.copy_(envs[0].targets)
    for e in envs:
        e.reset()
    ref = envs[0]
    for e in envs[1:]:
        assert torch.equal(e.grids, ref.grids) and torch.equal(e.stats, ref.stats)
    n_act = _n_act(ref, rep, shape)
    gen = torch.Generator(device=ref.device).manual_seed(5)
    steps = int(ref.max_iterations * 2.5) + 7
    for t in range(steps):
        act = torch.randint(0, n_act, (n,), generator=gen, device=ref.device, dtype=torch.int32)
        outs = []
        for path, e in zip(paths, envs):
            monkeypatch.setenv("PCGRL_STEP_PATH", path)
            r, d = e.step(act)
            outs.append((r.clone(), d.clone()))
        for (r, d), e, path in zip(outs[1:], envs[1:], paths[1:]):
            assert torch.equal(r, outs[0][0]), (path, t, int((r != outs[0][0]).sum()))
            assert torch.equal(d, outs[0][1]), (path, t)
            assert torch.equal(e.stats, ref.stats), (path, t, int((e.stats != ref.stats).any(dim=1).sum()))
            assert torch.equal(e.grids, ref.grids) and torch.equal(e.pos, ref.pos), (path, t)
            assert torch.equal(e.changes, ref.changes) and torch.equal(e.iteration, ref.iteration), (path, t)
            assert torch.equal(e.changed, ref.changed), (path, t)
        if t % 16 == 5 or t == steps - 1:
            for e in envs[2:]:
                fresh = e.compute_stats(e.maps, holes=e.holes) if e.holey else e.compute_stats(e.maps)
                assert torch.equal(fresh, e.stats), (t, int((fresh != e.stats).any(dim=1).sum()))
            if has_cache:      # the incremental paths keep the same cache rows (they may alternate on one shard)
                assert torch.equal(envs[2].cache, envs[3].cache) and torch.equal(envs[2].cache, envs[4].cache), t
    for e in envs:
        e.check_status()


@pytest.mark.parametrize("n,shape", [(30_000, (16, 16)), (60_000, (16, 16)), (400_000, (16, 16)), (400_000, (6, 9))])
def test_lanegroup_step_tiles_and_persistent_grid(n, shape, monkeypatch):
    """k_step_lanegroup picks 8 / 16 / 32 envs per warp by shard size and loops when the shard needs more warps than
    one wave holds: every variant must agree with the three-launch incremental path, and a shard may alternate
    between the two from step to step (same cache rows)."""
    envs = _envs("binary", "narrow", shape, n, ["inc", "lg"], max_board_scans=0.02)
    for e in envs:
        e.reset()
    a, b = envs
    gen = torch.Generator(device=a.device).manual_seed(9)
    for t in range(int(a.max_iterations * 2.2) + 3):
        act = torch.randint(0, 2, (n,), generator=gen, device=a.device, dtype=torch.int32)
        monkeypatch.setenv("PCGRL_STEP_PATH", "inc" if t % 5 != 4 else "lg")
        ra, da = a.step(act)
        ra, da = ra.clone(), da.clone()
        monkeypatch.setenv("PCGRL_STEP_PATH", "lg" if t % 7 != 6 else "inc")
        rb, db = b.step(act)
        assert torch.equal(ra, rb) and torch.equal(da, db), t
        assert torch.equal(a.stats, b.stats) and torch.equal(a.grids, b.grids) and torch.equal(a.cache, b.cache), t
    assert torch.equal(b.compute_stats(b.maps), b.stats)
    b.check_status()


def test_incremental_cache_is_consistent_with_the_grids(monkeypatch):
    """The cache row of every env holds the passable board of its CURRENT grid after resets and after steps, and a
    shard restored from state_dict continues bit-identically (the cache is part of the state)."""
    import control_pcgrl_b200 as P
    n = 4096
    cfg = P.make_config("binary", "narrow", map_shape=(16, 16), max_board_scans=0.3)
    env = P.BatchedPcgrlEnv(cfg, n, seed=2, auto_reset=True)
    assert env.cache is not None and env.cache_stride == 80
    env.reset()

    def board_of(maps):
        m = (maps.reshape(n, 256) == 0).to(torch.int64)              # tile 0 = empty = passable
        w = (m.reshape(n, 8, 32) << torch.arange(32, device=m.device)).sum(dim=2)   # bit y*16+x of word y//2
        return w.to(torch.int64)

    def cached_board():
        c = env.cache.view(torch.int32).reshape(n, 20)[:, :8].to(torch.int64) & 0xFFFFFFFF
        return c

    assert torch.equal(cached_board(), board_of(env.maps))
    gen = torch.Generator(device=env.device).manual_seed(0)
    for t in range(200):
        env.step(torch.randint(0, 2, (n,), generator=gen, device=env.device, dtype=torch.int32))
        if t % 25 == 0:
            assert torch.equal(cached_board(), board_of(env.maps)), t
    sd = env.state_dict()
    twin = P.BatchedPcgrlEnv(cfg, n, seed=99, auto_reset=True)
    twin.load_state_dict(sd)
    for t in range(120):
        a = torch.randint(0, 2, (n,), generator=gen, device=env.device, dtype=torch.int32)
        r0, _ = env.step(a)
        r1, _ = twin.step(a)
        assert torch.equal(r0, r1) and torch.equal(env.stats, twin.stats) and torch.equal(env.grids, twin.grids), t


def test_incremental_hand_built_maps():
    """Edits that merge, split, create and delete components on hand-built maps, including the component that holds
    the longest path (forces the re-sweep of the untouched components) -- each step checked against a fresh
    pcgrl_stats of the edited map."""
    import control_pcgrl_b200 as P
    cfg = P.make_config("binary", "wide", map_shape=(16, 16), obs_window=(16, 16))
    env = P.BatchedPcgrlEnv(cfg, 1, action_kind="wide_coords")
    g = np.ones((16, 16), dtype=np.int8)
    g[0, :] = 0           # a long corridor (path 15)
    g[2, 0:6] = 0         # a shorter one (path 5)
    g[4, 3] = 0           # an isolated cell
    g[6:9, 6:9] = 0       # a 3x3 room
    env.reset(grids=g[None])
    edits = [(1, 0, 0),    # join corridor 1 and corridor 2 through (1, 0)
             (0, 7, 1),    # cut the long corridor in two
             (0, 7, 0),    # and restore it
             (1, 0, 1),    # separate the two corridors again
             (4, 3, 1),    # delete the isolated cell
             (4, 3, 0),    # and bring it back
             (7, 7, 1),    # punch the room's centre (a ring)
             (0, 0, 1), (0, 1, 1), (0, 2, 1),   # eat the longest corridor from its first tile
             (15, 15, 0), (15, 14, 0), (14, 15, 0),  # grow a new component in the corner
             (5, 3, 0), (3, 3, 0),      # connect the isolated cell to corridor 2 and beyond
             (2, 3, 1)]                 # split corridor 2 (now a T) at the junction
    for y, x, v in edits:
        a = torch.tensor([[y, x, v]], dtype=torch.int32, device=env.device)
        env.step(a)
        fresh = env.compute_stats(env.maps)
        assert torch.equal(fresh, env.stats), ((y, x, v), fresh.tolist(), env.stats.tolist())
    env.check_status()


@pytest.mark.parametrize("rep,shape,controls,compact", [("narrow", (16, 16), None, True),
                                                        ("wide", (16, 16), ["regions", "path-length"], False),
                                                        ("turtle", (7, 5), None, True),
                                                        ("narrow", (3, 4), None, False),
                                                        ("narrow", (2, 16), None, True)])
def test_chunked_host_pipeline_equals_device_step(rep, shape, controls, compact, monkeypatch):
    """pcgrl_step_host's chunked pipeline (per chunk: upload, the three kernels of the incremental split path on one
    of the rotating compute streams, download) must give exactly what a whole-shard pcgrl_step gives, for every chunk
    count (ragged last chunk, chunks smaller than a warp's slice, up to the 64 work-list headers), across
    auto-resets, and interleaved with plain device steps on the same work-list headers."""
    import control_pcgrl_b200 as P
    n = 70_001
    kw = dict(obs_window=shape) if rep == "wide" else {}
    cfg = P.make_config("binary", rep, map_shape=shape, controls=controls, max_board_scans=0.05, **kw)
    a = P.BatchedPcgrlEnv(cfg, n, seed=3, auto_reset=True, compact_host_io=compact)
    b = P.BatchedPcgrlEnv(cfg, n, seed=3, auto_reset=True)
    assert a.cache is not None and a.worklist is not None
    if controls:
        g = torch.Generator(device=a.device).manual_seed(1)
        a.sample_uniform_targets(generator=g)
        b.targets.copy_(a.targets)
    a.reset()
    b.reset()
    n_act = _n_act(a, rep, shape)
    rng = np.random.default_rng(0)
    launches = a.lib.pcgrl_launch_count
    for t, chunks in enumerate(["2", "8", "5", "64", "3", "", "7", "1", "4", "16"] * 3):
        if chunks:
            monkeypatch.setenv("PCGRL_HOST_CHUNKS", chunks)
        else:
            monkeypatch.delenv("PCGRL_HOST_CHUNKS", raising=False)
        act = rng.integers(0, n_act, size=n).astype(a.action_shape_dtype()[1])
        l0 = launches()
        r, d, s = a.step_host(act)
        launched = launches() - l0
        if chunks not in ("1", ""):      # (the default is one chunk below 128 Ki envs: plain upload / step / download)
            n_ck = int(chunks)
            n_ck = -(-n // ((-(-n // n_ck) + 255) // 256 * 256))      # ragged: chunks of whole 256-env tiles
            # 3 kernels per chunk [+ the auto-reset launch]
            assert launched in (3 * n_ck, 3 * n_ck + 1), (chunks, launched)
        if t % 4 == 3:     # a plain device step in between (header 0 is shared by all paths)
            act2 = rng.integers(0, n_act, size=n).astype(np.int32)
            a.step(torch.from_numpy(act2.astype(a.action_shape_dtype()[1])).to(a.device))
            b.step(torch.from_numpy(act).to(b.device, dtype=torch.int32))
            b.step(torch.from_numpy(act2).to(b.device))
        else:
            rb, db = b.step(torch.from_numpy(act).to(b.device, dtype=torch.int32))
            np.testing.assert_array_equal(np.asarray(r), rb.cpu().numpy())
            np.testing.assert_array_equal(np.asarray(d).astype(bool), db.cpu().numpy().astype(bool))
        assert torch.equal(a.grids, b.grids) and torch.equal(a.stats, b.stats) and torch.equal(a.pos, b.pos)
        assert torch.equal(a.iteration, b.iteration) and torch.equal(a.changes, b.changes)
        assert torch.equal(a.cache, b.cache)
    a.check_status()
    fresh = a.compute_stats(a.maps)
    assert torch.equal(fresh, a.stats)


def test_one_shard_may_alternate_between_all_step_paths(monkeypatch):
    """The split paths hand their work list from step to step through alternating header words (the item counters);
    a shard that switches path from step to step -- three-launch incremental, three-launch from scratch, one-launch,
    lane groups, fused -- must keep giving the fused kernel's results, and the incremental cache must survive the
    steps that do not use it."""
    n = 40_000
    a, b = _envs("binary", "narrow", (16, 16), n, ["inc", "fused"], max_board_scans=0.05)
    a.reset()
    b.reset()
    gen = torch.Generator(device=a.device).manual_seed(4)
    order = ["inc", "split", "inc", "inc", "split", "split", "inc", "incfused", "inc", "lg", "inc", "fused", "inc", "split"]
    for t in range(3 * len(order) + int(a.max_iterations) + 2):
        act = torch.randint(0, 2, (n,), generator=gen, device=a.device, dtype=torch.int32)
        monkeypatch.setenv("PCGRL_STEP_PATH", order[t % len(order)])
        ra, da = a.step(act)
        ra, da = ra.clone(), da.clone()
        monkeypatch.setenv("PCGRL_STEP_PATH", "fused")
        rb, db = b.step(act)
        assert torch.equal(ra, rb) and torch.equal(da, db), (t, order[t % len(order)])
        assert torch.equal(a.stats, b.stats) and torch.equal(a.grids, b.grids), (t, order[t % len(order)])
    assert torch.equal(a.compute_stats(a.maps), a.stats)
    a.check_status()
