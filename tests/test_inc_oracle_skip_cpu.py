"""CPU: the incremental update with the skipped final sweep (tests/inc_oracle_skip.py, as BinaryIncMachine runs it)
against the from-scratch oracle and against the joint-sweep update (tests/inc_oracle_joint.py) at every edit:
regions, path-length AND the cache (P, F, m) must be equal, so that cache rows stay interchangeable between the step
paths -- and the skip must actually fire."""
import numpy as np
import pytest

from tests.inc_oracle_joint import IncBinaryJoint
from tests.inc_oracle_skip import IncBinarySkip
from tests.test_inc_oracle_cpu import _check


def _state(inc):
    return inc.P, inc.F, inc.m, inc.regions, inc.path


@pytest.mark.parametrize("shape", [(16, 16), (7, 5), (2, 16), (3, 4)])
@pytest.mark.parametrize("density", [0.3, 0.5, 0.75])
def test_skip_update_equals_from_scratch_and_joint_update(shape, density):
    h, w = shape
    rng = np.random.default_rng([h, w, int(density * 100)])
    grid = (rng.random(shape) < density).astype(np.int64)         # 1 = solid
    skip = IncBinarySkip(grid.tolist())
    ref = IncBinaryJoint(grid.tolist())
    n = 0
    for t in range(240):
        if t < 120:                                                # the narrow representation's scan order
            y, x = divmod(t % (h * w), w)
            if int(rng.integers(0, 2)) == grid[y, x]:
                continue
        else:
            y, x = int(rng.integers(0, h)), int(rng.integers(0, w))
        grid[y, x] ^= 1
        ref.flip(y, x)
        skip.flip(y, x)
        n += 1
        _check(skip, grid, (t, y, x))
        assert _state(skip) == _state(ref), (t, y, x)
    assert skip.skipped >= n // 5, (skip.skipped, n)


def test_skip_update_on_narrow_rollouts():
    """Long narrow-representation rollouts on 16x16 maps, the flagship workload's edit pattern: about half of all
    changed grids skip their final sweep."""
    rng = np.random.default_rng(12)
    n = skipped = 0
    for _ in range(6):
        grid = rng.integers(0, 2, (16, 16)).astype(np.int64)
        skip, ref = IncBinarySkip(grid.tolist()), IncBinaryJoint(grid.tolist())
        s0 = int(rng.integers(0, 256))
        for t in range(512):
            y, x = divmod((s0 + t) % 256, 16)
            v = int(rng.integers(0, 2))
            if v == grid[y, x]:
                continue
            grid[y, x] = v
            ref.flip(y, x)
            skip.flip(y, x)
            n += 1
            assert _state(skip) == _state(ref), (t, y, x)
        _check(skip, grid, "end")
        skipped += skip.skipped
    assert skipped >= 0.35 * n, (skipped, n)


def test_skip_boundary_hand_built():
    """The bound meets path-length exactly (skipped, tie: m stays in the old component), then exceeds it by one with
    an eccentricity one above path-length (swept, path-length and m move)."""
    g = np.ones((16, 16), dtype=np.int64)
    g[0, 0:9] = 0                                                  # corridor: path 8, holds m
    g[4, 2:5] = 0                                                  # an upside-down U, its first tile the corner (4, 2):
    g[5:8, 2] = 0                                                  # left arm 3 cells (4 with (8, 2))
    g[5:7, 4] = 0                                                  # right arm 2 cells
    skip, ref = IncBinarySkip(g.tolist()), IncBinaryJoint(g.tolist())
    assert skip.path == 8
    m0 = skip.m
    steps = [((8, 2), True, 8),     # e1 = 4, |C| - 1 = 8: bound 8 = path, lu = 8, skipped; m stays
             ((9, 2), False, 9),    # e1 = 5, lu = 9: swept, path and m move into the U
             ((9, 2), False, 8),    # m's component edited: the joint sweep, tie to the untouched corridor
             ((0, 4), False, 8)]    # cut the corridor that holds m: the U keeps path 8
    for (y, x), skipped, path in steps:
        before = skip.skipped
        g[y, x] ^= 1
        ref.flip(y, x)
        skip.flip(y, x)
        _check(skip, g, (y, x))
        assert _state(skip) == _state(ref), (y, x)
        assert (skip.skipped > before, skip.path) == (skipped, path), (y, x)
        if (y, x) == (8, 2):
            assert skip.m == m0
