"""CPU: the vectorised reference observation (oracle/obs_oracle.py) against the per-env loop functions of
oracle/pcgrl_oracle.py (cropped_onehot, full_onehot, static_builds_crop, target_channels), bit for bit after the
cast to every output dtype; and the case table of tests/test_gpu_observe.py against the writer variants."""
import itertools

import numpy as np
import pytest
import torch

from oracle import obs_oracle
from oracle import pcgrl_oracle as O

DTYPES = (torch.uint8, torch.float32, torch.float64)
# synthetic controlled metrics: (lo, hi) bounds with ranges that are not powers of two
BOUNDS = {"m0": (0, 136.0), "m1": (1, 7.5), "m2": (0, 38.5), "m3": (0, 1856)}
NAMES = list(BOUNDS)


def _reference(grid, pos, window, crop, n_tiles, static=None, ctrl=(), trg_row=None, stat_row=None):
    """One env through the loop functions, float64 [*window, C] with the map channels one-hot, and its tile codes."""
    hot = O.cropped_onehot(grid, pos, window, n_tiles) if crop else O.full_onehot(grid, n_tiles)
    codes = hot.argmax(axis=-1)[..., None].astype(np.float64)
    planes = []
    if ctrl:
        names = [NAMES[k] for k in ctrl]
        trgs = {NAMES[k]: (float(trg_row[k, 0]) if np.isnan(trg_row[k, 1])
                           else (float(trg_row[k, 0]), float(trg_row[k, 1]))) for k in ctrl}
        stats = {NAMES[k]: int(stat_row[k]) for k in ctrl}
        planes.append(O.target_channels(hot.shape[:-1], names, trgs, stats, BOUNDS))
    tail = [O.static_builds_crop(static, pos, window)[..., None]] if static is not None else []
    return np.concatenate(planes + [hot] + tail, axis=-1), np.concatenate(planes + [codes] + tail, axis=-1)


def _first_mismatch(got, want):
    bad = (got != want).nonzero()
    i = tuple(int(v) for v in bad[0])
    return f"env {i[0]} pixel {i[1:-1]} channel {i[-1]}: got {got[i].item()} want {want[i].item()}"


def _check(maps, pos, window, crop, n_tiles, static=None, ctrl=(), targets=None, stats=None):
    n = maps.shape[0]
    refs = [_reference(maps[e], pos[e], window, crop, n_tiles, None if static is None else static[e], ctrl,
                       None if targets is None else targets[e], None if stats is None else stats[e]) for e in range(n)]
    hot = torch.from_numpy(np.stack([r[0] for r in refs]))
    codes = torch.from_numpy(np.stack([r[1] for r in refs]))
    kw = dict(maps=torch.from_numpy(maps), pos=torch.from_numpy(pos), window=window, crop=crop, n_tiles=n_tiles,
              static_mask=None if static is None else torch.from_numpy(static))
    if ctrl:
        kw.update(targets=torch.from_numpy(targets), stats=torch.from_numpy(stats), ctrl_idx=list(ctrl),
                  ctrl_range=[abs(BOUNDS[NAMES[k]][1] - BOUNDS[NAMES[k]][0]) for k in ctrl])
    for dt in DTYPES:
        if ctrl and dt == torch.uint8:
            continue
        got, want = obs_oracle.observe(dtype=dt, **kw), hot.to(dt)
        assert got.dtype == dt and got.shape == want.shape, (dt, got.shape, want.shape)
        assert torch.equal(got, want), (dt, _first_mismatch(got, want))
    if not ctrl:
        got, want = obs_oracle.observe(dtype=torch.uint8, onehot=False, **kw), codes.to(torch.uint8)
        assert got.shape == want.shape and torch.equal(got, want), ("codes", _first_mismatch(got, want))
    return hot


def _batch(rng, shape, n_tiles, n_random=0):
    """Every position of the map once, then n_random random positions, each with its own random map."""
    every = np.array(list(itertools.product(*[range(d) for d in shape])), dtype=np.int32).reshape(-1, len(shape))
    rand = np.stack([rng.integers(0, d, n_random) for d in shape], axis=1).astype(np.int32)
    pos = np.concatenate([every, rand])
    maps = rng.integers(0, n_tiles, size=(len(pos), *shape)).astype(np.int8)
    return maps, pos


# windows smaller than the map, equal to it, 2x it and beyond 2x, odd and even (and mixed) extents
CASES_2D = [((5, 7), w) for w in [(3, 5), (2, 4), (5, 7), (10, 14), (9, 13), (13, 16), (11, 18), (4, 15)]] + \
           [((4, 4), w) for w in [(8, 8), (7, 7), (1, 1), (12, 9)]] + [((6, 3), (12, 6)), ((6, 3), (3, 9))]
CASES_3D = [((3, 4, 5), w) for w in [(6, 8, 10), (3, 5, 7), (2, 2, 4), (7, 9, 11), (8, 4, 6), (3, 4, 5)]] + \
           [((2, 3, 2), (5, 5, 5))]


@pytest.mark.parametrize("shape,window", CASES_2D + CASES_3D, ids=lambda v: "x".join(map(str, v)))
def test_crop_matches_loop_oracle(shape, window):
    rng = np.random.default_rng(sum(shape) * 131 + sum(window))
    for n_tiles in (2, 8) if len(shape) == 2 else (2, 3):
        maps, pos = _batch(rng, shape, n_tiles, n_random=12)
        hot = _check(maps, pos, window, True, n_tiles)
        assert hot.sum() == len(pos) * int(np.prod(window))


@pytest.mark.parametrize("shape", [(5, 7), (1, 9), (3, 4, 5), (2, 1, 3)])
def test_full_map_matches_loop_oracle(shape):
    rng = np.random.default_rng(len(shape) * 7 + shape[0])
    for n_tiles in (2, 5, 8):
        maps = rng.integers(0, n_tiles, size=(150, *shape)).astype(np.int8)
        _check(maps, np.zeros((150, len(shape)), np.int32), None, False, n_tiles)


@pytest.mark.parametrize("shape,window", [((5, 7), (10, 14)), ((5, 7), (9, 13)), ((5, 7), (4, 4)),
                                          ((5, 7), (13, 16)), ((4, 4), (3, 3)), ((3, 4, 5), (6, 8, 10)),
                                          ((3, 4, 5), (5, 7, 9)), ((3, 4, 5), (9, 11, 13))],
                         ids=lambda v: "x".join(map(str, v)))
def test_static_plane_matches_loop_oracle(shape, window):
    rng = np.random.default_rng(17 * sum(window))
    maps, pos = _batch(rng, shape, 3, n_random=20)
    static = (rng.random(maps.shape) < 0.3).astype(np.uint8)
    hot = _check(maps, pos, window, True, 3, static=static)
    st = hot[..., -1]
    # the border frame shows up as 1s, and a window reaching beyond it as 0s
    assert st.max() == 1 and st.min() == 0


def _targets(rng, n, tuple_every):
    """[n, K, 2] targets: (value, NaN), or a (lo, hi) range on every `tuple_every`-th env."""
    t = np.full((n, len(NAMES), 2), np.nan)
    for k, name in enumerate(NAMES):
        lo, hi = BOUNDS[name]
        t[:, k, 0] = rng.uniform(lo, hi, n)
        rows = np.arange(n) % tuple_every == 0 if tuple_every else np.zeros(n, bool)
        a = rng.integers(int(lo), int(hi), n).astype(np.float64)
        t[rows, k, 0] = a[rows]
        t[rows, k, 1] = a[rows] + rng.integers(1, 9, n)[rows]
    return t


@pytest.mark.parametrize("ctrl", [(1,), (0, 2), (3, 1)])
@pytest.mark.parametrize("tuple_every", [0, 1, 3])
@pytest.mark.parametrize("shape,window,static", [((5, 7), (10, 14), False), ((5, 7), (9, 9), True),
                                                 ((5, 7), None, False), ((3, 4, 5), (6, 8, 10), False)])
def test_control_planes_match_loop_oracle(ctrl, tuple_every, shape, window, static):
    rng = np.random.default_rng(len(ctrl) * 100 + tuple_every * 10 + len(shape))
    crop = window is not None
    maps, pos = _batch(rng, shape, 2, n_random=10)
    n = len(maps)
    stats = np.stack([rng.integers(0, int(BOUNDS[k][1]) + 3, n) for k in NAMES], axis=1).astype(np.int32)
    st = (rng.random(maps.shape) < 0.5).astype(np.uint8) if static else None
    hot = _check(maps, pos, window, crop, 2, static=st, ctrl=ctrl, targets=_targets(rng, n, tuple_every), stats=stats)
    assert hot.shape[-1] == 2 * len(ctrl) + (3 if crop else 2) + (1 if static else 0)


def test_rejects_fractional_planes_in_integer_output():
    maps = np.zeros((2, 4, 4), np.int8)
    kw = dict(maps=torch.from_numpy(maps), pos=torch.zeros((2, 2), dtype=torch.int32), window=(8, 8), n_tiles=2,
              targets=torch.zeros((1, 2, 2), dtype=torch.float64), stats=torch.zeros((2, 2), dtype=torch.int32),
              ctrl_idx=[0], ctrl_range=[10.0])
    with pytest.raises(ValueError):
        obs_oracle.observe(dtype=torch.uint8, **kw)
    with pytest.raises(ValueError):
        obs_oracle.observe(dtype=torch.float32, onehot=False, **kw)


def test_case_table_reaches_every_writer_variant():
    """Every variant of the observation writer is reached by at least one case of the GPU sweep (the labels come from
    the Python mirror of launch_vec in tests/test_gpu_observe.py)."""
    from tests import test_gpu_observe as G
    reached = set()
    for case in G.CASES:
        reached |= G.case_labels(case)
    missing = sorted(G.REQUIRED_LABELS - reached)
    assert not missing, missing
