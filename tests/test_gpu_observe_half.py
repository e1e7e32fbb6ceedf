"""GPU: float16 and bfloat16 observations (pcgrl_obs_args.out_kind 5 / 6).  Every element must be byte for byte the
float32 observation converted to the half type (round to nearest even), so everything here compares int16 views.

Every case of the float32 / uint8 writer suite (tests/test_gpu_observe.py::CASES) runs in both half types against the
reference observation in float32, converted: into observe()'s own allocation, into a sentinel-filled buffer at a
16-byte-aligned offset, and one element past it (the pixel-per-thread kernel); the guard bands must stay untouched.
half_variant() mirrors the 2-byte dispatch of launch_vec, and test_every_half_variant_is_reached checks that the cases
reach every 2-byte kernel.  The other tests cover double rounding of the target planes, holey maps, observe(env_ids),
lookahead / lookahead_all, PcgrlVectorEnv with its final observations, and the RLlib seam."""
import math

import numpy as np
import pytest
import torch

from oracle import obs_oracle
from tests.test_gpu_observe import CASES, N_TILES, Case, _make_env

HALF = (torch.float16, torch.bfloat16)
# a 2-byte group of the 3D maze's 30^3 window (162 000 bytes) still fits the stage: a 32^3 window does not
HALF_CASES = CASES + [Case("oversize_maze15_w32", "minecraft_3D_maze", "narrow", (15, 15, 15), (32, 32, 32), ())]


def half_variant(crop, shape, window, n_tiles, n_ctrl=0, static=False, holey=False, aligned=True):
    """(variant, G, GB) of a 2-byte one-hot observe() call.  Mirrors launch_vec in csrc/observe.cu for sizeof(T) == 2
    (group sizes, the row-mask flag `bits`, and the kernel choice) and must change with it."""
    if not aligned:
        return "scalar_unaligned", 0, 0
    d3 = len(shape) == 3
    o = tuple(window) if crop else tuple(shape)
    pix = math.prod(o)
    n_ch = 2 * n_ctrl + (n_tiles + 1 if crop else n_tiles) + (1 if static else 0)
    G = 1
    while (G * pix * n_ch * 2) % 16:
        G *= 2
    group_bytes = G * pix * n_ch * 2
    if group_bytes > 160 * 1024:
        return "scalar_oversize", G, 0
    GB = 1
    while GB * G * 2 <= 64 and GB * 2 * group_bytes <= 24 * 1024:
        GB *= 2
    bits = (crop and not d3 and n_tiles == 2 and shape[1] <= 16 and o[1] <= 32 and o[1] % 8 == 0 and not static and
            not holey and n_ctrl == 0 and n_ch == 3)
    last = o[-1]
    if bits:
        v = "bits8"
    elif not holey and not static and crop and d3 and o[2] == 14:
        v = "row14_7"
    else:
        v = "row0" if holey else "row4" if last % 4 == 0 else "row0"
    return v, G, GB


def _variant(case, aligned=True):
    crop = case.rep in ("narrow", "turtle")
    return half_variant(crop, case.shape, case.window, N_TILES[case.problem], len(case.controls or ()), case.static,
                        aligned=aligned)


def case_labels(case):
    quals = [q for q, on in (("3d", len(case.shape) == 3), ("ctrl", bool(case.controls)), ("nocrop", case.window is None),
                             ("static", case.static)) if on]
    v = _variant(case)[0]
    return {"scalar_unaligned", v} | {f"{v}/{q}" for q in quals}


REQUIRED = {"bits8", "row14_7", "row4", "row0", "scalar_unaligned", "scalar_oversize",
            "row4/3d", "row4/static", "row4/ctrl", "row4/nocrop", "row0/3d", "row0/static", "row0/ctrl", "row0/nocrop"}


def test_every_half_variant_is_reached():
    """CPU: the cases reach every 2-byte kernel launch_vec can pick, in its 3D / frozen-tile / control-plane /
    whole-map forms."""
    reached = set().union(*(case_labels(c) for c in HALF_CASES))
    assert REQUIRED <= reached, REQUIRED - reached


def _sizes(case, n_sm):
    """As tests/test_gpu_observe.py: partial groups and vector tails, and for the `big` cases enough envs that every CTA
    of the persistent staged writer takes at least two trips (at most 8 CTAs of 256 threads per SM)."""
    _, G, GB = _variant(case)
    sizes = sorted({1, 2, 7, 37, G + 1} | ({G - 1} if G > 1 else set()))
    return sizes, (2 * n_sm * 8 * max(GB, 1) * max(G, 1) + 3 if case.big else None)


def _reference(env, dtype):
    crop = env.representation in ("narrow", "turtle")
    return obs_oracle.observe(
        env.maps, env.pos[:, :env.ndim], env.obs_window if crop else None, crop, env.n_tiles,
        static_mask=env.static_tiles, targets=env.targets, stats=env.stats,
        ctrl_idx=[env.stat_names.index(k) for k in env.ctrl_metrics],
        ctrl_range=[env.param_ranges[k] for k in env.ctrl_metrics], dtype=torch.float32).to(dtype)


def _assert_same(got, want, what):
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype, want.dtype)
    g, w = got.view(torch.int16), want.view(torch.int16)
    if torch.equal(g, w):
        return
    i = tuple((g != w).nonzero()[0].tolist())
    raise AssertionError(f"{what}: first mismatch at {i}: got {got[i].item()} want {want[i].item()} "
                         f"({int((g != w).sum())} elements differ)")


GUARD = 64


def _observe_into_buffer(env, dtype, want, aligned, what, **kw):
    off, numel = GUARD + (0 if aligned else 1), want.numel()
    buf = torch.full((off + numel + GUARD,), float("nan"), dtype=dtype, device=env.device)
    view = buf[off:off + numel].view(want.shape)
    assert (view.data_ptr() % 16 == 0) == aligned
    got = env.observe(out=view, **kw)
    assert got.data_ptr() == view.data_ptr()
    _assert_same(view, want, what)
    for name, g in (("before", buf[:off]), ("after", buf[off + numel:])):
        assert bool(torch.isnan(g).all()), (what, f"guard band {name} the view was written")


@pytest.mark.gpu
@pytest.mark.parametrize("case", HALF_CASES, ids=[c.id for c in HALF_CASES])
def test_half_observe_matches_reference(case):
    sizes, big = _sizes(case, torch.cuda.get_device_properties(0).multi_processor_count)
    for n in sizes + ([big] if big else []):
        env = _make_env(case, n, seed=n)
        for dtype in HALF:
            what = f"{case.id} n={n} {dtype} [{_variant(case)[0]}]"
            want = _reference(env, dtype)
            assert want.shape == (n, *env.obs_shape())
            _assert_same(env.observe(dtype=dtype), want, what)
            _observe_into_buffer(env, dtype, want, True, what + " aligned buffer")
            if n != big:
                _observe_into_buffer(env, dtype, want, False, what + " unaligned buffer")
        del env


def _round_direct(x, mant):
    """x (a Python float) rounded ONCE to a binary float with `mant` fraction bits, nearest even (normal range)."""
    m, e = math.frexp(x)
    return round(m * 2.0 ** (mant + 1)) * 2.0 ** (e - mant - 1)


def _twice_differs(rng_val, dtype):
    """A target t whose plane t / rng_val, rounded straight to `dtype`, differs from the value rounded to float32
    first: the float32 value sits exactly on a tie of the half type, the double just beside it."""
    mant = 10 if dtype == torch.float16 else 7
    for k in range(1, 4000):
        tie = 0.5 + (2 * k + 1) * 2.0 ** (-mant - 2)          # halfway between two neighbours in [0.5, 1)
        for t in (tie * rng_val + d * 2.0 ** -30 for d in (-3, -2, -1, 1, 2, 3)):
            x = t / rng_val
            f32 = float(np.float32(x))
            if f32 == tie and x != tie:
                twice = torch.tensor([f32], dtype=torch.float32).to(dtype).item()
                if twice != _round_direct(x, mant):
                    return t, twice, _round_direct(x, mant)
    raise AssertionError("no double-rounding target found")


@pytest.mark.gpu
def test_target_planes_round_through_float32():
    """A target plane is round_half((float)(t / range)): on a tie of the float32 value the direct rounding of the
    double differs, and the writers (staged, and pixel-per-thread through an unaligned buffer) must give the former."""
    import control_pcgrl_b200 as P
    for rep, window in (("wide", None), ("narrow", (32, 32))):
        cfg = P.make_config("binary", rep, obs_window=window, controls=["path-length"])
        env = P.BatchedPcgrlEnv(cfg, 8, seed=2)
        env.reset()
        col = env.stat_names.index("path-length")
        rng_val = float(env.param_ranges["path-length"])
        for dtype in HALF:
            t, twice, direct = _twice_differs(rng_val, dtype)
            assert twice != direct
            env.targets[:, col, 0] = t
            env.targets[:, col, 1] = float("nan")
            want = env.observe(dtype=torch.float32).to(dtype)
            assert float(want[0].reshape(-1, want.shape[-1])[0, 0]) == twice
            for aligned in (True, False):
                _observe_into_buffer(env, dtype, want, aligned, f"{rep} {dtype} aligned={aligned}")
            got = env.observe(dtype=dtype)
            _assert_same(got, want, f"{rep} {dtype}")
            assert float(got[0].reshape(-1, got.shape[-1])[0, 0]) == twice


@pytest.mark.gpu
@pytest.mark.parametrize("problem,rep,shape,window", [
    ("binary_holey", "narrow", (16, 16), None), ("binary_holey", "turtle", (9, 13), (15, 15)),
    ("binary_holey", "wide", (16, 16), None), ("minecraft_3D_holey_maze", "narrow", (7, 7, 7), None)])
def test_holey_half_equals_float32_converted(problem, rep, shape, window):
    import control_pcgrl_b200 as P
    kw = {"obs_window": window} if window else {}
    env = P.BatchedPcgrlEnv(P.make_config(problem, rep, map_shape=shape, **kw), 37, seed=4,
                            action_kind="wide_coords" if rep == "wide" else None)
    env.reset()
    f32 = env.observe(dtype=torch.float32)
    for dtype in HALF:
        want = f32.to(dtype)
        _assert_same(env.observe(dtype=dtype), want, f"{problem} {rep} {dtype}")
        _observe_into_buffer(env, dtype, want, False, f"{problem} {rep} {dtype} unaligned")
        ids = [36, 0, 5, 5, 17]
        _assert_same(env.observe(dtype=dtype, env_ids=ids), want[ids], f"{problem} {rep} {dtype} env_ids")


@pytest.mark.gpu
def test_observe_env_ids_half():
    """Rows in any order with repeats; the device index guard writes nothing through a bad index and sets bit 64."""
    import control_pcgrl_b200 as P
    for problem, rep, kw in (("binary", "narrow", {}), ("zelda", "turtle", {}),
                             ("binary", "wide", {"controls": ["regions", "path-length"]})):
        env = P.BatchedPcgrlEnv(P.make_config(problem, rep, **kw), 300, seed=3)
        if env.ctrl_metrics:
            env.sample_uniform_targets()
        env.reset()
        for dtype in HALF:
            full = env.observe(dtype=torch.float32).to(dtype)
            ids = torch.tensor([299, 3, 3, 0, 150, 3, 298], dtype=torch.int32, device=env.device)
            _assert_same(env.observe(dtype=dtype, env_ids=ids), full[ids.long()], f"{problem} {rep} {dtype}")
            big = torch.randint(0, 300, (5000,), dtype=torch.int32, device=env.device)
            _assert_same(env.observe(dtype=dtype, env_ids=big), full[big.long()], f"{problem} {rep} {dtype} 5000")
            # an index outside the shard, past the host check: bit 64, the other rows are right
            bad = torch.tensor([1, 300, 2], dtype=torch.int32, device=env.device)
            env.status.zero_()
            out = env._observe_envs(bad, dtype=dtype)
            torch.cuda.synchronize()
            assert int(env.status.item()) & 64
            _assert_same(out[[0, 2]], full[[1, 2]], f"{problem} {rep} {dtype} guard")
            env.status.zero_()


@pytest.mark.gpu
def test_unsupported_dtypes_raise_before_anything_runs():
    import control_pcgrl_b200 as P
    env = P.BatchedPcgrlEnv(P.make_config("binary", "narrow"), 4, seed=1)
    env.reset()
    before = env.lib.pcgrl_launch_count()
    for dt in (torch.int16, torch.float8_e4m3fn, torch.int32):
        with pytest.raises(TypeError):
            env.observe(dtype=dt)
        with pytest.raises(TypeError):
            env.observe(out=torch.empty((4, *env.obs_shape()), dtype=dt, device=env.device))
        with pytest.raises(TypeError):
            env.lookahead(torch.zeros(4, dtype=torch.int32, device=env.device), obs_dtype=dt)
        with pytest.raises(TypeError):
            env.lookahead_all(obs_dtype=dt)
    assert env.lib.pcgrl_launch_count() == before


@pytest.mark.gpu
@pytest.mark.parametrize("problem,rep,shape,cfg,env_kw,agent", [
    ("binary", "narrow", (16, 16), {}, {}, 0),                                   # search cache: incremental path
    ("zelda", "turtle", (7, 11), {}, {}, 0),                                     # generic path
    ("binary", "narrow", (16, 16), {"controls": ["regions", "path-length"]}, {}, 0),
    ("zelda", "turtle", (7, 11), {"show_agents": True}, {"n_agents": 3}, 2),     # occupancy plane in the same dtype
], ids=["binary_narrow_cached", "zelda_turtle_generic", "binary_narrow_controls", "zelda_show_agents"])
def test_lookahead_half_equals_float32_converted(problem, rep, shape, cfg, env_kw, agent):
    import control_pcgrl_b200 as P
    n = 97
    env = P.BatchedPcgrlEnv(P.make_config(problem, rep, map_shape=shape, **cfg), n, seed=6, **env_kw)
    if env.ctrl_metrics:
        env.sample_uniform_targets()
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(6)
    A = env.n_discrete_actions()
    for _ in range(5):
        env.step(torch.randint(0, A, (n,), generator=g, device=env.device, dtype=torch.int32), agent=agent)
    ids = torch.randint(0, n, (300,), generator=g, device=env.device, dtype=torch.int32)
    acts = torch.randint(0, A, (300,), generator=g, device=env.device, dtype=torch.int32)
    ref = env.lookahead(acts, env_ids=ids, agent=agent, obs_dtype=torch.float32)
    ref_all = env.lookahead_all(agent=agent, obs_dtype=torch.float32)
    for dtype in HALF:
        got = env.lookahead(acts, env_ids=ids, agent=agent, obs_dtype=dtype)
        assert torch.equal(got[0].view(torch.int32), ref[0].view(torch.int32))
        assert all(torch.equal(a, b) for a, b in zip(got[1:4], ref[1:4]))
        _assert_same(got[4], ref[4].to(dtype), f"{problem} {rep} lookahead {dtype}")
        out = torch.empty_like(got[4])
        got2 = env.lookahead(acts, env_ids=ids, agent=agent, obs_out=out)
        assert got2[4].data_ptr() == out.data_ptr()
        _assert_same(out, ref[4].to(dtype), f"{problem} {rep} lookahead obs_out {dtype}")
        all_ = env.lookahead_all(agent=agent, obs_dtype=dtype)
        assert all(torch.equal(a, b) for a, b in zip(all_[1:4], ref_all[1:4]))
        _assert_same(all_[4], ref_all[4].to(dtype), f"{problem} {rep} lookahead_all {dtype}")


@pytest.mark.gpu
def test_lookahead_all_half_chunks_by_element_size(monkeypatch):
    """lookahead_all bounds its chunks by observation bytes: 2-byte elements fit twice the candidates of float32."""
    import control_pcgrl_b200 as P
    env = P.BatchedPcgrlEnv(P.make_config("binary", "narrow"), 40, seed=8)
    env.reset()
    whole = env.lookahead_all(obs_dtype=torch.bfloat16)
    per_obs = math.prod(env.obs_shape()) * 2
    monkeypatch.setattr(type(env), "LOOKAHEAD_OBS_CHUNK_BYTES", per_obs * 6)    # three envs of 2 actions per chunk
    calls = []
    real = type(env)._lookahead_obs

    def spy(self, a, rows, m, *rest):
        calls.append(m)
        return real(self, a, rows, m, *rest)
    monkeypatch.setattr(type(env), "_lookahead_obs", spy)
    chunked = env.lookahead_all(obs_dtype=torch.bfloat16)
    assert max(calls) == 6 and sum(calls) == 80
    _assert_same(chunked[4], whole[4], "chunked")


def _same_draws(fn_a, fn_b):
    """fn_a(), then fn_b() from the same global CUDA RNG state: sample_uniform_targets draws from it."""
    state = torch.cuda.get_rng_state()
    ra = fn_a()
    torch.cuda.set_rng_state(state)
    return ra, fn_b()


def _vector_pair(dtype, shards, n=96):
    import control_pcgrl_b200 as P
    from control_pcgrl_b200.vector_env import PcgrlVectorEnv
    cfg = P.make_config("binary", "wide", max_board_scans=0.03, controls=["regions", "path-length"])
    return (PcgrlVectorEnv(cfg, n, seed=5, shards=shards, obs_dtype=dtype, uniform_targets=True),
            PcgrlVectorEnv(cfg, n, seed=5, shards=shards, obs_dtype=torch.float32, uniform_targets=True))


@pytest.mark.gpu
@pytest.mark.parametrize("shards", [1, 2])
@pytest.mark.parametrize("dtype", HALF, ids=["f16", "bf16"])
def test_vector_env_half_with_controls(dtype, shards):
    """PcgrlVectorEnv on binary-wide + controls against a float32 twin with the same seed and actions: observations
    and final observations are the float32 ones converted, rewards and dones identical."""
    venv, twin = _vector_pair(dtype, shards)
    (obs, _), (ref, _) = _same_draws(venv.reset, twin.reset)
    assert obs.dtype == dtype
    _assert_same(obs, ref.to(dtype), "reset")
    n = venv.num_envs
    gen = torch.Generator(device=obs.device).manual_seed(1)
    ends = 0
    for t in range(60):
        act = torch.randint(0, venv.single_action_space.n, (n,), generator=gen, device=obs.device, dtype=torch.int32)
        (obs, rew, _, done, info), (ref, rew2, _, done2, info2) = _same_draws(lambda: venv.step(act),
                                                                              lambda: twin.step(act))
        assert torch.equal(rew.view(torch.int32), rew2.view(torch.int32)) and torch.equal(done, done2), t
        _assert_same(obs, ref.to(dtype), f"step {t}")
        assert set(info) == set(info2)
        if info:
            ends += 1
            assert torch.equal(info["final_idx"], info2["final_idx"])
            assert info["final_obs"].dtype == dtype
            _assert_same(info["final_obs"], info2["final_obs"].to(dtype), f"final_obs {t}")
    assert ends >= 2


@pytest.mark.gpu
def test_rllib_seam_float16():
    """make_rllib_vector_env(obs_dtype=np.float16): float16 host rows equal to the float32 seam's, converted."""
    import control_pcgrl_b200 as P
    n = 64
    cfg = P.make_config("binary", "narrow", max_board_scans=0.05, change_percentage=0.2, controls=["regions"])
    half = P.make_rllib_vector_env(cfg, n, seed=4, obs_dtype=np.float16)
    full = P.make_rllib_vector_env(cfg, n, seed=4, obs_dtype=np.float32)
    assert half.observation_space.dtype == np.float16
    (o16, _), (o32, _) = _same_draws(half.vector_reset, full.vector_reset)
    assert o16[0].dtype == np.float16
    np.testing.assert_array_equal(np.stack(o16).view(np.int16), np.stack(o32).astype(np.float16).view(np.int16))
    rng = np.random.default_rng(0)
    finished = 0
    for t in range(40):
        acts = [int(a) for a in rng.integers(0, 2, size=n)]
        o16, r16, _, d16, _ = half.vector_step(acts)
        o32, r32, _, d32, _ = full.vector_step(acts)
        assert r16 == r32 and d16 == d32, t
        np.testing.assert_array_equal(np.stack(o16).view(np.int16), np.stack(o32).astype(np.float16).view(np.int16))
        for i in np.flatnonzero(d16):
            a, _ = half.reset_at(int(i))
            b, _ = full.reset_at(int(i))
            np.testing.assert_array_equal(a.view(np.int16), b.astype(np.float16).view(np.int16))
            finished += 1
    assert finished >= n
