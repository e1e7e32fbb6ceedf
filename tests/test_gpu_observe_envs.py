"""The observation of a list of envs (pcgrl_observe_envs, BatchedPcgrlEnv.observe(env_ids=...)): for every case of the
writer sweep in tests/test_gpu_observe.py, in every kind the case runs, observe(env_ids=idx) must equal observe()[idx]
and the reference observation's rows idx, written into a sentinel-filled buffer at an aligned and at an unaligned
offset (the pixel kernel) with its guard bands intact.  Index patterns: one env, all envs ascending and reversed,
random with duplicates, G - 1 and G + 1 rows, and for the `big` cases more rows than the persistent staged grid covers
in one trip (every CTA takes two).  Then the forms the sweep has no case for (holey maps, a second agent's crop with
the occupancy plane), the host / device index validation, and the ABI's argument checks."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import obs_oracle
from tests.test_gpu_observe import (CASES, GUARD, KINDS, REQUIRED_LABELS, _assert_same, _make_env, _reference,
                                    _variant, case_labels)

N_ENVS = 37


def test_cases_reach_every_writer_variant():
    """CPU: the sweep below runs every case of tests/test_gpu_observe.py, so it reaches every writer label."""
    reached = set()
    for case in CASES:
        reached |= case_labels(case)
    assert not sorted(REQUIRED_LABELS - reached)


def _patterns(n, G, rng):
    pats = {"one": np.array([n // 2]), "ascending": np.arange(n), "reversed": np.arange(n)[::-1].copy(),
            "random_dups": rng.integers(0, n, n + 5)}
    for m in sorted({max(G - 1, 1), G + 1}):
        pats[f"M={m}"] = rng.integers(0, n, m)
    return pats


def _into_buffer(env, kind, idx, want, aligned, what):
    dtype, onehot = KINDS[kind]
    off, numel = GUARD + (0 if aligned else 1), want.numel()
    buf = torch.empty(off + numel + GUARD, dtype=dtype, device=env.device)
    buf.fill_(0xA5 if dtype == torch.uint8 else float("nan"))
    view = buf[off:off + numel].view(want.shape)
    assert (view.data_ptr() % 16 == 0) == aligned
    got = env.observe(out=view, onehot=onehot, env_ids=idx)
    assert got.data_ptr() == view.data_ptr()
    _assert_same(view, want, what)
    for name, g in (("before", buf[:off]), ("after", buf[off + numel:])):
        intact = (g == 0xA5).all() if dtype == torch.uint8 else torch.isnan(g).all()
        assert bool(intact), (what, f"guard band {name} the view was written")


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_observe_envs_matches_full_rows(case):
    n = N_ENVS
    env = _make_env(case, n, seed=11)
    rng = np.random.default_rng(7)
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    for kind in case.kinds:
        dtype, onehot = KINDS[kind]
        v, G, GB = _variant(case, kind)
        full = env.observe(dtype=dtype, onehot=onehot)
        ref = _reference(env, kind)
        _assert_same(full, ref, f"{case.id} {kind} full")
        pats = _patterns(n, G, rng)
        if case.big == kind:          # every CTA of the persistent staged grid takes at least two trips
            pats["big"] = rng.integers(0, n, 2 * n_sm * 8 * GB * G + 3)
        for name, idx in pats.items():
            what = f"{case.id} {kind} [{v}] env_ids={name}"
            t = torch.from_numpy(idx).to(env.device)
            want = full[t]
            _assert_same(env.observe(dtype=dtype, onehot=onehot, env_ids=t), want, what)
            if name == "random_dups":
                _assert_same(env.observe(dtype=dtype, onehot=onehot, env_ids=idx), ref[t], what + " vs reference")
            _into_buffer(env, kind, t, want, True, what + " aligned buffer")
            if name != "big":
                _into_buffer(env, kind, t, want, False, what + " unaligned buffer")


@pytest.mark.gpu
@pytest.mark.parametrize("problem,rep", [("binary_holey", "narrow"), ("binary_holey", "wide"),
                                         ("minecraft_3D_holey_maze", "narrow"), ("minecraft_3D_dungeon_holey", "narrow"),
                                         ("minecraft_3D_holey_maze", "wide")])
def test_observe_envs_holey(problem, rep):
    """The bordered maps with their holes: 2D through the staged general path, 3D through the pixel kernel."""
    import control_pcgrl_b200 as P
    n = 41
    kw = dict(map_shape=(5, 5, 5), obs_window=(6, 8, 10)) if problem != "binary_holey" else {}
    env = P.BatchedPcgrlEnv(P.make_config(problem, rep, **kw), n, seed=3,
                            action_kind="wide_coords" if rep == "wide" else None)
    env.reset()
    if rep == "narrow":
        for i, d in enumerate(env.map_shape):
            env.pos[:, i] = torch.randint(0, d, (n,), device=env.device, dtype=torch.int32)
    idx = torch.from_numpy(np.random.default_rng(1).integers(0, n, 2 * n + 1)).to(env.device)
    for dtype in (torch.uint8, torch.float32):
        full = env.observe(dtype=dtype)
        _assert_same(env.observe(dtype=dtype, env_ids=idx), full[idx], f"{problem} {rep} {dtype}")
        _assert_same(env.observe(dtype=dtype, env_ids=idx.flip(0)), full[idx.flip(0)], f"{problem} {rep} {dtype} rev")
    full = env.observe(onehot=False)
    _assert_same(env.observe(onehot=False, env_ids=idx), full[idx], f"{problem} {rep} codes")


@pytest.mark.gpu
def test_observe_envs_second_agent_and_occupancy_plane():
    import control_pcgrl_b200 as P
    n = 29
    cfg = P.make_config("binary", "turtle", map_shape=(16, 16), obs_window=(32, 32))
    cfg.multiagent.n_agents = 3
    env = P.BatchedPcgrlEnv(cfg, n, seed=5)
    env.reset()
    cfg2 = P.make_config("binary", "turtle", map_shape=(16, 16), obs_window=(32, 32))
    cfg2.multiagent.n_agents = 3
    cfg2.show_agents = True
    shown = P.BatchedPcgrlEnv(cfg2, n, seed=5)
    shown.reset()
    assert shown.show_agents and not env.show_agents
    idx = torch.from_numpy(np.random.default_rng(2).integers(0, n, n + 7)).to(env.device)
    for e in (env, shown):
        for agent in (1, 2):
            for dtype, onehot in ((torch.uint8, True), (torch.float32, True), (torch.uint8, False)):
                full = e.observe(dtype=dtype, onehot=onehot, agent=agent)
                got = e.observe(dtype=dtype, onehot=onehot, agent=agent, env_ids=idx)
                _assert_same(got, full[idx], f"show_agents={e.show_agents} agent {agent} {dtype} {onehot}")
                out = torch.empty_like(full[idx])
                assert e.observe(out=out, onehot=onehot, agent=agent, env_ids=idx) is out
                _assert_same(out, full[idx], "into out")
    want = obs_oracle.observe(env.maps[idx], env.agent_pos[1, idx, :2], (32, 32), True, env.n_tiles, dtype=torch.uint8)
    _assert_same(env.observe(dtype=torch.uint8, agent=1, env_ids=idx), want, "agent 1 vs reference")


@pytest.mark.gpu
def test_observe_envs_rejects_bad_indices_and_writes_nothing():
    import control_pcgrl_b200 as P
    n = 12
    env = P.BatchedPcgrlEnv(P.make_config("binary", "narrow"), n, seed=1)
    env.reset()
    lib = env.lib
    dev = env.device
    bad = [[-1], [0, n], [n + 100], np.array([[0, 1]]), np.array([0.0, 1.0]), 3]
    bad += [torch.tensor(b) for b in ([-1], [0, n], [[0, 1]])]
    bad += [torch.tensor(b, device=dev) for b in ([-1], [0, n], [n, 0, 1], [[0, 1]])]
    bad += [torch.tensor([0.0, 1.0], device=dev)]
    for ids in bad:
        out = torch.full((2, *env.obs_shape()), 0xA5, dtype=torch.uint8, device=dev)
        before = lib.pcgrl_launch_count()
        with pytest.raises(IndexError):
            env.observe(out=out, env_ids=ids)
        assert lib.pcgrl_launch_count() == before, ids
        assert bool((out == 0xA5).all()), ids
    # n_idx == 0: an empty result, nothing launched
    for ids in ([], np.zeros(0, dtype=np.int64), torch.zeros(0, dtype=torch.int64, device=dev)):
        before = lib.pcgrl_launch_count()
        got = env.observe(dtype=torch.uint8, env_ids=ids)
        assert tuple(got.shape) == (0, *env.obs_shape()) and got.dtype == torch.uint8
        assert lib.pcgrl_launch_count() == before
    # the device entry point with n_idx == 0 is a no-op too, and the status word stays clear
    env.check_status()
    torch.cuda.synchronize()
    assert int(env.status.item()) == 0
    # uint8 / int16 indices are integers too
    full = env.observe(dtype=torch.uint8)
    for ids in (np.array([3, 1, 3], dtype=np.uint8), torch.tensor([3, 1, 3], dtype=torch.int16, device=dev)):
        _assert_same(env.observe(dtype=torch.uint8, env_ids=ids), full[[3, 1, 3]], str(ids))


@pytest.mark.gpu
def test_abi_observe_envs_zero_rows_launch_nothing():
    import control_pcgrl_b200 as P
    env = P.BatchedPcgrlEnv(P.make_config("binary", "narrow"), 4, seed=1)
    env.reset()
    from control_pcgrl_b200 import _lib
    oa = _lib.ObsArgs()
    oa.crop, oa.out_kind = 1, 0
    oa.obs_dims[0], oa.obs_dims[1], oa.obs_dims[2] = 32, 32, 1
    out = torch.empty(16, dtype=torch.uint8, device=env.device)
    oa.out = out.data_ptr()
    before = env.lib.pcgrl_launch_count()
    assert env.lib.pcgrl_observe_envs(env._cc, env._st, oa, None, 0, None) == 0
    assert env.lib.pcgrl_launch_count() == before


def _cfg():
    from control_pcgrl_b200 import _lib
    c = _lib.Config()
    c.abi_version = _lib.PCGRL_ABI_VERSION
    c.problem, c.representation, c.action_kind = _lib.PROB_IDS["binary"], _lib.REP_IDS["narrow"], _lib.ACT_INT32
    c.ndim, c.dims[0], c.dims[1] = 2, 16, 16
    c.n_tiles, c.n_stats, c.max_iterations, c.max_changes = 2, 2, 769, -1
    return c


def test_abi_observe_envs_argument_errors_cpu():
    """CPU: NULL config / state / obs args / env_idx (n_idx > 0) and n_idx < 0 are PCGRL_E_ARG, checked before any
    pointer is dereferenced; without a device a valid call is PCGRL_E_CUDA (no CPU fallback)."""
    from control_pcgrl_b200 import _lib
    lib = _lib.load()
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    st, oa = _lib.State(), _lib.ObsArgs()
    st.n_envs, st.grids, st.pos = 4, 0x10000, 0x20000          # never dereferenced on these paths
    oa.crop, oa.out_kind, oa.out = 1, 0, 0x30000
    oa.obs_dims[0], oa.obs_dims[1], oa.obs_dims[2] = 32, 32, 1
    idx = (ctypes.c_int32 * 2)(0, 1)
    E_ARG, E_CUDA = -1, -2
    assert lib.pcgrl_observe_envs(None, st, oa, idx, 2, None) == E_ARG
    assert lib.pcgrl_observe_envs(c, None, oa, idx, 2, None) == E_ARG
    assert lib.pcgrl_observe_envs(c, st, None, idx, 2, None) == E_ARG
    assert lib.pcgrl_observe_envs(c, st, oa, None, 2, None) == E_ARG
    assert b"env_idx" in lib.pcgrl_last_error()
    assert lib.pcgrl_observe_envs(c, st, oa, idx, -1, None) == E_ARG
    assert b"n_idx" in lib.pcgrl_last_error()
    if torch.cuda.is_available():
        return              # the call below would launch on fake pointers
    assert lib.pcgrl_observe_envs(c, st, oa, idx, 2, None) == E_CUDA
