"""GPU: BatchedPcgrlEnv.update (pcgrl_update, k_update) -- Representation.update without get_stats.

Twin envs with the same config and seed are driven with the same actions, one by step() and one by update(): maps,
positions, n_step, frozen-tile masks and `changed` must agree bit for bit after every call, while the update env's
counters, stats, reward, done, records, work list and search cache stay exactly as they were.  A sample of envs is
checked against the reference's rep_update, and the stats of the final maps against the step twin's.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SMALL_PRIME = 1009


def _big_n():
    """Envs enough for every CTA of k_update's persistent grid to make at least two trips: a trip covers at most
    2048 envs per SM (2048 resident threads per SM; a cellular CTA of 256 threads covers 256 envs)."""
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 2048 + 1   # 606,209 on 148 SMs


# name -> (problem, rep, map_shape, make_config extras, BatchedPcgrlEnv extras)
CASES = {
    "binary-narrow": ("binary", "narrow", (16, 16), {}, {}),
    "binary-turtle": ("binary", "turtle", (16, 16), {}, {}),
    "binary-wide-flat": ("binary", "wide", (16, 16), {"obs_window": (16, 16)}, {}),
    "binary-wide-coords": ("binary", "wide", (16, 16), {"obs_window": (16, 16)}, {"action_kind": "wide_coords"}),
    "binary-narrow-64": ("binary", "narrow", (64, 64), {}, {}),
    "zelda-turtle": ("zelda", "turtle", (7, 11), {}, {}),
    "binary_holey-narrow": ("binary_holey", "narrow", (16, 16), {}, {}),
    "sokoban-ca-tiles": ("sokoban", "cellular", (5, 5), {}, {"action_kind": "ca_tiles"}),
    "sokoban-ca-logits": ("sokoban", "cellular", (5, 5), {}, {}),
    "sokoban-ca-logits-ties": ("sokoban", "cellular", (5, 5), {}, {}),
    "smb-ca-tiles": ("smb", "cellular", (116, 16), {}, {"action_kind": "ca_tiles"}),
    "smb-ca-logits": ("smb", "cellular", (116, 16), {}, {}),
    "smb-ca-logits-ties": ("smb", "cellular", (116, 16), {}, {}),
    "binary-ca-logits": ("binary", "cellular", (16, 16), {}, {}),
    "binary-ca-logits-ties": ("binary", "cellular", (16, 16), {}, {}),
    "mc3d-narrow": ("minecraft_3D_maze", "narrow", (14, 14, 14), {}, {}),
    "mc3d-turtle": ("minecraft_3D_maze", "turtle", (14, 14, 14), {}, {}),
    "mc3d-wide-coords": ("minecraft_3D_maze", "wide", (14, 14, 14), {"obs_window": (14, 14, 14)},
                         {"action_kind": "wide_coords"}),
    "mc3d_holey_maze-narrow": ("minecraft_3D_holey_maze", "narrow", (7, 7, 7), {}, {}),
    "mc3d_dungeon_holey-narrow": ("minecraft_3D_dungeon_holey", "narrow", (7, 7, 7), {}, {}),
    "binary-patch": ("binary", "narrow", (16, 16), {"act_window": (3, 2)}, {}),
    "mc3d-patch": ("minecraft_3D_maze", "narrow", (14, 14, 14), {"act_window": (2, 3, 2)}, {}),
    "binary-static-narrow": ("binary", "narrow", (16, 16),
                             {"static_tile_wrapper": True, "static_prob": 1.0, "n_static_walls": 2}, {}),
    "binary-static-turtle": ("binary", "turtle", (16, 16),
                             {"static_tile_wrapper": True, "static_prob": 1.0, "n_static_walls": 2}, {}),
    "binary-multiagent-turtle": ("binary", "turtle", (8, 8), {"n_agents": 3}, {}),
    "binary-narrow-compact": ("binary", "narrow", (16, 16), {}, {"compact_host_io": True}),
}
# the cheap cases also run a shard on which every CTA of the persistent grid loops at least twice
BIG = {"binary-narrow", "binary-static-narrow", "binary-ca-logits", "sokoban-ca-tiles", "sokoban-ca-logits-ties",
       "binary-narrow-compact"}
PARAMS = [(c, n) for c in CASES for n in (1, SMALL_PRIME, "big") if n != "big" or c in BIG]


def _bits(t):
    """Raw bytes of a tensor: targets hold NaN (scalar targets), which torch.equal never calls equal."""
    return t.contiguous().view(torch.uint8)


UNTOUCHED = ("iteration", "changes", "stats", "reward", "done", "records", "cache", "worklist", "targets", "holes")


def _twins(case, n, seed=7):
    import control_pcgrl_b200 as P
    problem, rep, shape, cfg_kw, env_kw = CASES[case]
    cfg_kw = dict(cfg_kw)
    n_agents = cfg_kw.pop("n_agents", None)
    cells = int(np.prod(shape))
    cfg = P.make_config(problem, rep, map_shape=shape, max_board_scans=12 / cells, **cfg_kw)
    if n_agents:
        cfg.multiagent.n_agents = n_agents
    return [P.BatchedPcgrlEnv(cfg, n, seed=seed, auto_reset=False, **env_kw) for _ in range(2)]


def _actions(env, case, gen):
    """One random action batch of env's layout.  Cellular batches leave about a quarter of the maps as they are
    (changed = 0); the *-ties cases draw logits from {0, 1, 2} so that most cells tie between channels."""
    n, dev, C = env.n_envs, env.device, env.n_tiles
    shape, _, tdt = env._action_layout()
    ak = env.action_kind
    if ak in ("int32", "wide_flat"):
        hi = {"narrow": C, "turtle": 4 + C}.get(env.representation, env.obs_window[0] * env.obs_window[1] * C)
        return torch.randint(0, hi, shape, generator=gen, device=dev).to(tdt)
    if ak == "wide_coords":
        cols = [torch.randint(0, d, (n, 1), generator=gen, device=dev) for d in env.map_shape]
        cols.append(torch.randint(0, C, (n, 1), generator=gen, device=dev))
        return torch.cat(cols, dim=1).to(torch.int32)
    if ak == "patch":
        return torch.randint(0, C, shape, generator=gen, device=dev).to(torch.int32)
    keep = torch.rand(n, generator=gen, device=dev) < 0.25
    cur = env.grids[:, :env.cells].long()
    if ak == "ca_tiles":
        t = torch.zeros(shape, dtype=torch.int8, device=dev)      # padding bytes stay 0, as in the grids
        new = torch.randint(0, C, (n, env.cells), generator=gen, device=dev)
        t[:, :env.cells] = torch.where(keep[:, None], cur, new).to(torch.int8)
        return t
    if case.endswith("-ties"):
        lg = torch.randint(0, 3, (n, C, env.cells), generator=gen, device=dev).float()
    else:
        lg = torch.randn((n, C, env.cells), generator=gen, device=dev)
    onehot = torch.nn.functional.one_hot(cur, C).permute(0, 2, 1).float()      # argmax = the current map
    return torch.where(keep[:, None, None], onehot, lg).reshape(shape).contiguous()


def _oracle_update(env, grid, pos, n_step, static, act):
    """oracle.pcgrl_oracle.rep_update on one env; returns (grid, pos, n_step, change)."""
    from oracle import pcgrl_oracle as O
    nd, shape = env.ndim, env.map_shape
    coords = O.narrow_coords(shape) if env.act_window is None else O.multiaction_coords(shape, env.act_window)
    state = {"pos": [int(v) for v in pos[:nd]], "n_step": int(n_step), "coords": coords,
             "act_window": env.act_window, "static": static}
    ak = env.action_kind
    if ak in ("int32",):
        a = int(act)
    elif ak == "wide_flat":
        a = O.actionmap_unravel(int(act), env.obs_window[0], env.obs_window[1], env.n_tiles)
    elif ak == "wide_coords":
        a = [int(v) for v in act]
    elif ak == "patch":
        a = np.asarray(act)
    elif ak == "ca_tiles":
        a = np.asarray(act[:env.cells]).reshape(shape).astype(np.int64)
    else:
        a = np.asarray(act).reshape(env.n_tiles, *shape)
    g = grid.astype(np.int64).copy()
    change = O.rep_update(env.representation, g, state, a)
    return g, state["pos"], state["n_step"], change


@pytest.mark.parametrize("case,n", PARAMS)
def test_update_equals_step_and_reference(case, n):
    if n == "big":
        n = _big_n()
    a, b = _twins(case, n)                      # a: step(), b: update()
    a.reset()
    b.reset()
    assert torch.equal(a.grids, b.grids) and torch.equal(a.agent_pos, b.agent_pos)
    A = max(b.n_agents, 1)
    gen = torch.Generator(device=a.device).manual_seed(3)
    rng = np.random.default_rng(0)
    sample = np.sort(rng.choice(n, size=min(n, 64), replace=False))
    sample_t = torch.from_numpy(sample).to(a.device)
    nd = b.ndim
    steps = int(b.max_iterations) + 3
    assert steps > b.max_iterations
    for t in range(steps):
        agent = t % A
        act = _actions(b, case, gen)
        before = {k: _bits(getattr(b, k)).clone() for k in UNTOUCHED if getattr(b, k) is not None}
        s_grid = b.maps[sample_t].cpu().numpy()
        s_pos = b.agent_pos[agent][sample_t].cpu().numpy()
        s_nstep = b.n_step[sample_t].cpu().numpy()
        s_static = None if b.static_mask is None else b.static_tiles[sample_t].cpu().numpy()
        s_act = act.reshape(n, -1)[sample_t].cpu().numpy() if act.dim() > 1 else act[sample_t].cpu().numpy()

        a.step(act, agent=agent)
        ch = b.update(act, agent=agent)
        torch.cuda.synchronize()
        assert ch.dtype == torch.uint8 and tuple(ch.shape) == (n,)
        assert torch.equal(a.grids, b.grids), (t, int((a.grids != b.grids).any(dim=1).sum()))
        assert torch.equal(a.agent_pos, b.agent_pos), t
        assert torch.equal(a.n_step, b.n_step), t
        if b.static_mask is not None:
            assert torch.equal(a.static_mask, b.static_mask), t
        assert torch.equal(ch, a.changed), (t, int((ch != a.changed).sum()))
        for k, v in before.items():
            assert torch.equal(_bits(getattr(b, k)), v), (k, t)

        g_now = b.maps[sample_t].cpu().numpy()
        p_now = b.agent_pos[agent][sample_t].cpu().numpy()
        n_now = b.n_step[sample_t].cpu().numpy()
        c_now = ch[sample_t].cpu().numpy()
        for j in range(len(sample)):
            g, p, ns, change = _oracle_update(b, s_grid[j], s_pos[j], s_nstep[j],
                                              None if s_static is None else s_static[j].astype(np.int64), s_act[j])
            assert np.array_equal(g_now[j], g), (t, int(sample[j]))
            assert p_now[j][:nd].tolist() == list(p), (t, int(sample[j]))
            assert int(n_now[j]) == int(ns), (t, int(sample[j]))
            assert int(c_now[j]) == int(change), (t, int(sample[j]))
    assert int(a.iteration.min()) > a.max_iterations          # the step twin ran past the end of its episode
    b.check_status()

    # end of the episode: stats of the updated maps = what the step twin computed along the way
    fresh = b.compute_stats(b.maps, holes=b.holes)
    cols = [k for k, s in enumerate(b.stat_names)
            if not (b.problem == "minecraft_3D_holey_maze" and s in ("path-length", "_next-path-length"))]
    assert torch.equal(fresh[:, cols], a.stats[:, cols]), int((fresh[:, cols] != a.stats[:, cols]).any(dim=1).sum())


def _guard_env(controls, n=257, seed=5):
    import control_pcgrl_b200 as P
    cfg = P.make_config("binary", "narrow", map_shape=(16, 16), controls=controls, max_board_scans=0.2)
    return P.BatchedPcgrlEnv(cfg, n, seed=seed)


def test_stale_guard():
    import control_pcgrl_b200 as P
    n = 257
    gen = torch.Generator(device="cuda").manual_seed(0)
    b = _guard_env(["regions", "path-length"])
    c = _guard_env(["regions", "path-length"])               # the same resets and steps, no update()
    assert b.cache is not None
    b.reset()
    c.reset()
    x = torch.randint(0, 2, (n,), generator=gen, device=b.device, dtype=torch.int32)
    launches = b.lib.pcgrl_launch_count
    l0 = launches()
    b.update(x)
    assert launches() - l0 == 1
    with pytest.raises(RuntimeError, match="reset"):
        b.step(x)
    with pytest.raises(RuntimeError, match="reset"):
        b.step_agents(x[:, None].contiguous())
    with pytest.raises(RuntimeError, match="reset"):
        b.step_host(x.cpu().numpy())
    with pytest.raises(RuntimeError, match="reset"):
        b.observe()                                              # control planes read stats
    assert launches() - l0 == 1                                  # the guards launched nothing

    # the flag travels with a checkpoint; a checkpoint without it loads as fresh
    sd = b.state_dict()
    assert sd["_stats_stale"] is True
    d = _guard_env(["regions", "path-length"])
    d.load_state_dict(sd)
    with pytest.raises(RuntimeError, match="reset"):
        d.step(x)
    sd.pop("_stats_stale")
    d.load_state_dict(sd)
    d.observe()

    mask = (torch.arange(n, device=b.device) % 3 == 0).to(torch.uint8)
    b.reset(mask=mask)
    c.reset(mask=mask)
    with pytest.raises(RuntimeError, match="reset"):
        b.step(x)
    b.reset()
    c.reset()
    for _ in range(3):
        y = torch.randint(0, 2, (n,), generator=gen, device=b.device, dtype=torch.int32)
        rb, db = b.step(y)
        rc, dc = c.step(y)
        assert torch.equal(rb, rc) and torch.equal(db, dc)
        assert torch.equal(b.stats, c.stats) and torch.equal(b.grids, c.grids) and torch.equal(b.cache, c.cache)
    assert torch.equal(b.observe(), c.observe())

    # map-only observations keep working after update(): they equal the step twin's
    u, s = _guard_env(None), _guard_env(None)
    u.reset()
    s.reset()
    for dtype in (torch.uint8, torch.float32):
        y = torch.randint(0, 2, (n,), generator=gen, device=u.device, dtype=torch.int32)
        u.update(y)
        s.step(y)
        assert torch.equal(u.observe(dtype=dtype), s.observe(dtype=dtype))
    assert torch.equal(u.observe(onehot=False), s.observe(onehot=False))
    assert isinstance(u, P.BatchedPcgrlEnv)


def test_invalid_update_action_sets_status():
    b = _guard_env(None)
    b.reset()
    x = torch.zeros(b.n_envs, dtype=torch.int32, device=b.device)
    x[17] = 7                                                    # binary has tiles 0 / 1
    g0 = b.grids[17].clone()
    ch = b.update(x)
    assert int(ch[17]) == 0 and torch.equal(b.grids[17], g0)   # ignored, as step ignores it
    with pytest.raises(ValueError):
        b.check_status()
    b.update(torch.zeros_like(x))
    b.check_status()
