"""GPU: every variant of the observation writer (csrc/observe.cu) against the vectorised reference observation
(oracle/obs_oracle.py, itself pinned on the per-env loop oracle by tests/test_obs_oracle_cpu.py).

Each case builds a BatchedPcgrlEnv, resets it, steps a few random actions (so that the stats, and with them the
control planes, are not trivial), puts the crop centres on corners, edges and random cells, and compares
env.observe() with obs_oracle.observe() of the same maps / positions / targets / stats / frozen-tile masks with
torch.equal: into observe()'s own allocation, and into a sentinel-filled buffer at a 16-byte-aligned and at an
unaligned offset, whose guard bands must stay untouched.  Batch sizes leave groups partly filled and the vector copy
with a tail; the `big` cases run enough envs for every CTA of the persistent staged writer to take two trips."""
import math
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import obs_oracle

pytestmark = pytest.mark.gpu

A_B_VARS = ("PCGRL_OBSERVE_SCALAR", "PCGRL_OBSERVE_NO_BITS", "PCGRL_OBSERVE_NO_ROW32", "PCGRL_OBSERVE_ROW22",
            "PCGRL_OBSERVE_ROW14")
KINDS = {"u8": (torch.uint8, True), "f32": (torch.float32, True), "f64": (torch.float64, True),
         "codes": (torch.uint8, False)}
ELEM = {"u8": 1, "codes": 1, "f32": 4, "f64": 8}


def writer_variant(kind, crop, shape, window, n_tiles, n_ctrl=0, static=False, env=(), aligned=True):
    """(variant, G, GB) the observation writer takes for one observe() call.

    This mirrors launch_observe / launch_vec in csrc/observe.cu (the dispatch at lines 495-560, the scalar-kernel
    switch at line 627, and the pack3 / pack1 / bits flags at the top of k_observe_staged) and must change with them.
    Nothing checks it against that code automatically: review it line by line when the dispatch changes.
    (The occupancy query's per_sm < 1 fallback is not mirrored; no case here comes near it.)"""
    env = dict(env)
    if "PCGRL_OBSERVE_SCALAR" in env:
        return "scalar_env", 0, 0
    if not aligned:
        return "scalar_unaligned", 0, 0
    size, raw, d3 = ELEM[kind], kind == "codes", len(shape) == 3
    o = tuple(window) if crop else tuple(shape)
    pix = math.prod(o)
    n_map_ch = 1 if raw else (n_tiles + 1 if crop else n_tiles)
    n_ch = 2 * n_ctrl + n_map_ch + (1 if static else 0)
    E = pix * n_ch
    G = 1
    while (G * E * size) % 16:
        G *= 2
    group_bytes = G * E * size
    if group_bytes > 160 * 1024:
        return "scalar_oversize", G, 0
    GB = 1
    while GB * G * 2 <= 64 and GB * 2 * group_bytes <= 24 * 1024:
        GB *= 2
    bits = (size == 1 and crop and not d3 and n_tiles == 2 and shape[1] <= 16 and o[1] <= 32 and o[1] % 8 == 0 and
            not static and n_ctrl == 0 and n_ch == (1 if raw else 3) and "PCGRL_OBSERVE_NO_BITS" not in env)
    last = o[-1]
    rown = 8 if size == 1 and last % 8 == 0 else (4 if last % 4 == 0 else 0)
    if size == 1 and rown == 0 and o[1] == 22 and not d3 and not static and crop:
        r22 = int(env.get("PCGRL_OBSERVE_ROW22", 11))
        rown = r22 if r22 in (11, 22) else rown
    if size == 1 and rown == 0 and d3 and o[2] == 14 and not static and crop:
        r14 = int(env.get("PCGRL_OBSERVE_ROW14", 7))
        rown = r14 if r14 in (7, 14) else rown
    if bits and rown == 8 and o[1] == 32 and not d3 and not static and crop and "PCGRL_OBSERVE_NO_ROW32" not in env:
        rown = 32
    r8 = rown in (8, 32)
    pack3 = size == 1 and r8 and not static and n_ch == 3 and not raw and n_ctrl == 0
    pack1 = size == 1 and r8 and not static and n_ch == 1 and raw and n_ctrl == 0
    if rown == 32:
        v = "row32"
    elif rown == 8:
        v = "row8_bits" if bits and (pack3 or pack1) else \
            "row8_pack3" if pack3 else "row8_pack1" if pack1 else "row8_generic"
    else:
        v = {0: "row0", 4: "row4", 11: "row22_11", 22: "row22_22", 7: "row14_7", 14: "row14_14"}[rown]
    return v, G, GB


Case = namedtuple("Case", "id problem rep shape window kinds env controls static big",
                  defaults=((), None, False, None))
U8C = ("u8", "codes")
ALL4 = ("u8", "f32", "f64", "codes")
CASES = [
    # staged, a whole 32-pixel window row per thread from row bit masks (two-tile maps <= 16 wide, any height)
    Case("row32_binary16", "binary", "narrow", (16, 16), (32, 32), U8C, big="u8"),
    Case("row32_binary40x16", "binary", "narrow", (40, 16), (32, 32), U8C),
    Case("row32_binary16x5", "binary", "narrow", (16, 5), (32, 32), U8C),
    Case("row32_binary9x13_odd_height", "binary", "turtle", (9, 13), (15, 32), U8C),
    # staged, 8 pixels per thread from row bit masks: windows smaller than the map, 24 wide, 32 wide without ROW32
    Case("bits_binary16_w8", "binary", "narrow", (16, 16), (8, 8), U8C),
    Case("bits_binary16_w24", "binary", "narrow", (16, 16), (24, 24), U8C),
    Case("bits_binary9x13_w16x24", "binary", "turtle", (9, 13), (16, 24), U8C),
    Case("bits_binary16_no_row32", "binary", "narrow", (16, 16), (32, 32), U8C, env={"PCGRL_OBSERVE_NO_ROW32": "1"}),
    # staged, 8 packed records per thread without bit masks (whole groups outside the map: constant records)
    Case("pack_binary20x24_w48", "binary", "narrow", (20, 24), (48, 48), U8C),
    Case("pack_binary16_no_bits", "binary", "narrow", (16, 16), (32, 32), U8C, env={"PCGRL_OBSERVE_NO_BITS": "1"}),
    Case("pack_binary64_default_window", "binary", "narrow", (64, 64), (32, 32), U8C),
    # staged, 8 pixels per thread, one store per pixel
    Case("generic8_zelda_w24", "zelda", "narrow", (7, 11), (24, 24), ("u8", "f32", "codes")),
    Case("generic8_smb", "smb", "narrow", (116, 16), (32, 32), U8C),
    Case("nocrop_binary_wide", "binary", "wide", (16, 16), None, ALL4),
    # 22-wide u8 windows: 11 (default) or 22 pixels per thread
    Case("row22_zelda", "zelda", "narrow", (7, 11), (22, 22), U8C, big="u8"),
    Case("row22_zelda_whole_row", "zelda", "turtle", (7, 11), (22, 22), U8C, env={"PCGRL_OBSERVE_ROW22": "22"}),
    Case("row22_off_zelda", "zelda", "narrow", (7, 11), (22, 22), U8C, env={"PCGRL_OBSERVE_ROW22": "0"}),
    Case("row22_binary16", "binary", "narrow", (16, 16), (22, 22), U8C),
    Case("row22_sokoban5", "sokoban", "narrow", (5, 5), (22, 22), U8C),
    Case("row22_zelda30_map_wider", "zelda", "narrow", (30, 30), (22, 22), U8C),
    # 3D crops whose last window axis is 14: 7 (default) or 14 pixels per thread
    Case("row14_maze14", "minecraft_3D_maze", "narrow", (14, 14, 14), (14, 14, 14), U8C, big="u8"),
    Case("row14_maze14_whole_row", "minecraft_3D_maze", "turtle", (14, 14, 14), (14, 14, 14), U8C,
         env={"PCGRL_OBSERVE_ROW14": "14"}),
    Case("row14_maze7", "minecraft_3D_maze", "narrow", (7, 7, 7), (14, 14, 14), U8C),
    Case("row14_maze5x9x7", "minecraft_3D_maze", "narrow", (5, 9, 7), (10, 18, 14), U8C),
    # 3D, 8 pixels per thread (packed one-hot / codes), 4 per thread in f32 / f64
    Case("rown8_maze3d", "minecraft_3D_maze", "turtle", (6, 7, 8), (12, 14, 16), ALL4),
    Case("nocrop_maze_wide_6x7x8", "minecraft_3D_maze", "wide", (6, 7, 8), None, ("u8", "f32", "codes")),
    # 4 pixels per thread
    Case("rown4_mc2d", "minecraft_2D_maze", "narrow", (14, 14), (28, 28), U8C),
    Case("rown4_binary16_float", "binary", "narrow", (16, 16), (32, 32), ("f32", "f64"), big="f32"),
    # general path (last window axis not a multiple of 4): odd windows are off-centre
    Case("odd_binary16_w15", "binary", "narrow", (16, 16), (15, 15), ALL4),
    Case("odd_binary16_w21", "binary", "narrow", (16, 16), (21, 21), U8C),
    Case("odd_zelda_w21", "zelda", "narrow", (7, 11), (21, 21), ("u8", "f64", "codes")),
    Case("odd_maze6_w9", "minecraft_3D_maze", "narrow", (6, 6, 6), (9, 9, 9), ALL4),
    Case("general_binary_turtle", "binary", "turtle", (9, 13), (18, 26), ("u8", "f32", "codes")),
    # frozen-tile plane
    Case("static_binary16", "binary", "narrow", (16, 16), (32, 32), ("u8", "f32", "f64"), static=True, big="u8"),
    Case("static_zelda", "zelda", "narrow", (7, 11), (22, 22), ("u8", "f32", "f64"), static=True),
    Case("static_binary_odd", "binary", "turtle", (9, 13), (17, 17), ("u8", "f32"), static=True),
    Case("static_maze3d", "minecraft_3D_maze", "narrow", (6, 7, 8), (12, 14, 16), ("u8", "f32"), static=True),
    # whole map, no crop
    Case("nocrop_zelda_wide", "zelda", "wide", (7, 11), None, ALL4),
    Case("nocrop_sokoban_cellular", "sokoban", "cellular", (5, 5), None, ALL4),
    Case("nocrop_maze_wide6", "minecraft_3D_maze", "wide", (6, 6, 6), None, ALL4),
    # control planes (per-env sampled targets, range targets on every third env)
    Case("ctrl_binary_wide", "binary", "wide", (16, 16), None, ("f32", "f64"), controls=("regions", "path-length")),
    Case("ctrl_binary_narrow", "binary", "narrow", (16, 16), (32, 32), ("f32", "f64"), controls=("path-length",)),
    Case("ctrl_zelda_static", "zelda", "narrow", (7, 11), (22, 22), ("f32", "f64"),
         controls=("nearest-enemy", "path-length"), static=True),
    # the one-thread-per-pixel kernel: forced, and for groups too large for the stage (3D maze's default 30^3 window)
    Case("scalar_binary16", "binary", "narrow", (16, 16), (32, 32), ALL4, env={"PCGRL_OBSERVE_SCALAR": "1"}),
    Case("scalar_maze_odd", "minecraft_3D_maze", "narrow", (6, 7, 8), (9, 9, 9), ("u8", "f32", "codes"),
         env={"PCGRL_OBSERVE_SCALAR": "1"}),
    Case("oversize_maze15", "minecraft_3D_maze", "narrow", (15, 15, 15), (30, 30, 30), ("u8", "f32", "f64")),
]
# every dispatch target of launch_vec, the 3D / frozen-tile / whole-map / control-plane forms of the staged paths,
# and the three ways into the scalar kernel
REQUIRED_LABELS = {
    "row32", "row8_bits", "row8_pack3", "row8_pack1", "row8_generic", "row22_11", "row22_22", "row14_7", "row14_14",
    "row4", "row0", "row8_pack3/3d", "row8_pack1/3d", "row8_generic/3d", "row4/3d", "row0/3d",
    "row8_generic/static", "row4/static", "row0/static", "row8_generic/3d/static", "row4/3d/static",
    "row8_generic/nocrop", "row8_generic/3d/nocrop", "row0/3d/nocrop", "row4/ctrl", "row4/ctrl/nocrop",
    "row0/ctrl/static", "scalar_env", "scalar_unaligned", "scalar_oversize",
}
N_TILES = {"binary": 2, "zelda": 8, "sokoban": 5, "smb": 7, "minecraft_2D_maze": 2, "minecraft_3D_maze": 2}


def _variant(case, kind, aligned=True):
    crop = case.rep in ("narrow", "turtle")
    return writer_variant(kind, crop, case.shape, case.window, N_TILES[case.problem], len(case.controls or ()),
                          case.static, case.env, aligned)


def case_labels(case):
    """The variant labels a case reaches: the bare variant, each qualifier (3d / static / nocrop / ctrl) on its own,
    all of them together, and the unaligned-buffer fallback every case also runs."""
    quals = [q for q, on in (("3d", len(case.shape) == 3), ("ctrl", bool(case.controls)), ("nocrop", case.window is None),
                             ("static", case.static)) if on]
    out = {"scalar_unaligned"}
    for kind in case.kinds:
        v = _variant(case, kind)[0]
        out |= {v, "/".join([v] + quals)} | {f"{v}/{q}" for q in quals}
    return out


def _sizes(case, n_sm):
    """1, 2, G - 1, G + 1 and two odd primes; for the `big` cases also n >= 2 * n_sm * 8 * GB * G (at most 8 CTAs of
    256 threads fit on an SM, so every CTA of the persistent grid takes at least two trips) plus an odd tail."""
    G = max(_variant(case, k)[1] for k in case.kinds)
    sizes = sorted({1, 2, 7, 37, G + 1} | ({G - 1} if G > 1 else set()))
    big = None
    if case.big:
        _, g, gb = _variant(case, case.big)
        big = 2 * n_sm * 8 * gb * g + 3
    return sizes, big


def _make_env(case, n, seed):
    import control_pcgrl_b200 as P
    kw = dict(obs_window=case.window or case.shape)
    if case.controls:
        kw["controls"] = list(case.controls)
    if case.static:
        kw.update(static_tile_wrapper=True, static_prob=0.3)
    env = P.BatchedPcgrlEnv(P.make_config(case.problem, case.rep, map_shape=case.shape, **kw), n, seed=seed)
    g = torch.Generator(device=env.device).manual_seed(seed)
    if case.controls:
        env.sample_uniform_targets(generator=g)
        lo, hi = env.cond_bounds[case.controls[0]]
        env.set_trgs({case.controls[0]: (lo + 1, (lo + hi) / 3)}, env_ids=torch.arange(0, n, 3, device=env.device))
    env.reset()
    # a few random steps: the stats (and the control planes) leave their reset values
    rep, nt = env.representation, env.n_tiles
    for _ in range(3):
        if rep == "cellular":
            a = torch.randn((n, nt * env.cells), generator=g, device=env.device)
        else:
            n_act = {"narrow": nt, "turtle": 4 + nt}.get(rep, env.obs_window[0] * env.obs_window[1] * nt)
            a = torch.randint(0, n_act, (n,), generator=g, device=env.device, dtype=env._action_layout()[2])
        env.step(a)
    if case.static:   # frozen tiles independent of the draw at reset, on about a third of the cells
        m = torch.rand((n, env.cells), generator=g, device=env.device) < 0.35
        env.static_mask[:, :env.cells] = m.to(torch.uint8)
    if case.window is not None:
        env.pos[:, :env.ndim] = torch.from_numpy(_positions(n, case.shape, seed)).to(env.device)
    return env


def _positions(n, shape, seed):
    """Crop centres: every corner, then cells on every face / edge, then random cells."""
    rng = np.random.default_rng(seed)
    nd = len(shape)
    pos = np.stack([rng.integers(0, d, n) for d in shape], axis=1)
    for e in range(n):
        if e < 2 ** nd:
            pos[e] = [(d - 1) * ((e >> i) & 1) for i, d in enumerate(shape)]
        elif e < 2 ** nd + 2 * nd:
            ax, hi = divmod(e - 2 ** nd, 2)
            pos[e, ax] = shape[ax] - 1 if hi else 0
    return pos.astype(np.int32)


def _reference(env, kind):
    dtype, onehot = KINDS[kind]
    crop = env.representation in ("narrow", "turtle")
    return obs_oracle.observe(
        env.maps, env.pos[:, :env.ndim], env.obs_window if crop else None, crop, env.n_tiles,
        static_mask=env.static_tiles, targets=env.targets, stats=env.stats,
        ctrl_idx=[env.stat_names.index(k) for k in env.ctrl_metrics],
        ctrl_range=[env.param_ranges[k] for k in env.ctrl_metrics], dtype=dtype, onehot=onehot)


def _assert_same(got, want, what):
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype)
    if torch.equal(got, want):
        return
    bad = (got != want).nonzero()[0].tolist()
    i = tuple(bad)
    raise AssertionError(f"{what}: first mismatch at env {i[0]} pixel {i[1:-1]} channel {i[-1]}: "
                         f"got {got[i].item()} want {want[i].item()} ({int((got != want).sum())} elements differ)")


GUARD = 64   # elements: a 16-byte multiple for every dtype


def _observe_into_buffer(env, kind, want, aligned, what):
    """observe() into a view of a larger sentinel-filled buffer (the slice of a rollout buffer a trainer hands over),
    at a 16-byte-aligned offset or one element past it; the guard bands around the view must stay untouched."""
    dtype, onehot = KINDS[kind]
    off, numel = GUARD + (0 if aligned else 1), want.numel()
    buf = torch.empty(off + numel + GUARD, dtype=dtype, device=env.device)
    buf.fill_(0xA5 if dtype == torch.uint8 else float("nan"))
    view = buf[off:off + numel].view(want.shape)
    assert (view.data_ptr() % 16 == 0) == aligned
    got = env.observe(out=view, onehot=onehot)
    assert got.data_ptr() == view.data_ptr()
    _assert_same(view, want, what)
    for name, g in (("before", buf[:off]), ("after", buf[off + numel:])):
        intact = (g == 0xA5).all() if dtype == torch.uint8 else torch.isnan(g).all()
        assert bool(intact), (what, f"guard band {name} the view was written")


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_observe_matches_reference(case, monkeypatch):
    for v in A_B_VARS:
        monkeypatch.delenv(v, raising=False)
    for k, v in dict(case.env).items():
        monkeypatch.setenv(k, v)
    sizes, big = _sizes(case, torch.cuda.get_device_properties(0).multi_processor_count)
    for n in sizes + ([big] if big else []):
        env = _make_env(case, n, seed=n)
        for kind in ((case.big,) if n == big else case.kinds):
            dtype, onehot = KINDS[kind]
            what = f"{case.id} n={n} {kind} [{_variant(case, kind)[0]}]"
            want = _reference(env, kind)
            assert want.shape == (n, *env.obs_shape(onehot))
            _assert_same(env.observe(dtype=dtype, onehot=onehot), want, what)
            _observe_into_buffer(env, kind, want, True, what + " aligned buffer")
            if n != big:
                _observe_into_buffer(env, kind, want, False, what + " unaligned buffer")
        del env


def test_rejections_write_nothing():
    """uint8 one-hot and tile codes cannot hold the fractional control planes: both raise before anything is
    written."""
    from control_pcgrl_b200 import _lib
    case = Case("ctrl", "binary", "narrow", (16, 16), (32, 32), ("f32",), controls=("path-length",))
    env = _make_env(case, 5, seed=3)
    for onehot, exc in ((True, _lib.PcgrlError), (False, ValueError)):
        out = torch.full((5, *env.obs_shape(onehot)), 0xA5, dtype=torch.uint8, device=env.device)
        with pytest.raises(exc):
            env.observe(out=out, onehot=onehot)
        assert bool((out == 0xA5).all()), onehot
    with pytest.raises(_lib.PcgrlError):
        env.observe(dtype=torch.uint8)


def test_second_agent_sees_its_own_crop():
    """Multi-agent turtle: observe(agent=1) is the crop around agent 1's position."""
    import control_pcgrl_b200 as P
    n = 37
    env = P.BatchedPcgrlEnv(P.make_config("binary", "turtle", map_shape=(16, 16), obs_window=(32, 32)), n, seed=5,
                            n_agents=2)
    env.reset()
    assert not env.show_agents
    env.agent_pos[1, :, :2] = torch.from_numpy(_positions(n, (16, 16), 5)).to(env.device)
    for kind in ("u8", "f32", "codes"):
        dtype, onehot = KINDS[kind]
        want = obs_oracle.observe(env.maps, env.agent_pos[1, :, :2], (32, 32), True, env.n_tiles, dtype=dtype,
                                  onehot=onehot)
        _assert_same(env.observe(dtype=dtype, onehot=onehot, agent=1), want, f"agent 1 {kind}")
        assert not torch.equal(env.agent_pos[0], env.agent_pos[1])
