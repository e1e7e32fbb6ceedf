"""CPU: the incremental update as BinaryIncMachine runs it (tests/inc_oracle_joint.py: one joint final sweep, isolated
cells counted next to the edited cell only) against the from-scratch oracle at every edit, and against
oracle/inc_oracle.py's two-sweep update, kept as the reference: regions, path-length AND the cache (P, F, m) must be
equal after every edit, so that cache rows stay interchangeable between the step paths."""
import numpy as np
import pytest

from oracle.inc_oracle import IncBinary
from tests.inc_oracle_joint import IncBinaryJoint
from tests.test_inc_oracle_cpu import _check


def _state(inc):
    return inc.P, inc.F, inc.m, inc.regions, inc.path


@pytest.mark.parametrize("shape", [(16, 16), (10, 10), (7, 5), (3, 4), (2, 16), (1, 9), (16, 3), (15, 16)])
@pytest.mark.parametrize("density", [0.3, 0.5, 0.75])
def test_joint_update_equals_from_scratch_and_two_sweep_update(shape, density):
    rng = np.random.default_rng(hash((shape, density, "joint")) & 0xFFFF)
    h, w = shape
    grid = (rng.random(shape) < density).astype(np.int64)         # 1 = solid
    joint = IncBinaryJoint(grid.tolist())
    ref = IncBinary(grid.tolist())
    for t in range(240):
        if t < 80:                                                 # the narrow representation's scan order
            y, x = divmod(t % (h * w), w)
            if int(rng.integers(0, 2)) == grid[y, x]:
                continue
        else:
            y, x = int(rng.integers(0, h)), int(rng.integers(0, w))
        grid[y, x] ^= 1
        ref.flip(y, x)
        joint.flip(y, x)
        _check(joint, grid, (t, y, x))
        assert _state(joint) == _state(ref), (t, y, x)


def test_joint_update_ties_and_isolated_cells():
    g = np.ones((16, 16), dtype=np.int64)
    g[0, :8] = 0                                                   # corridor, path 7
    g[4, :8] = 0                                                   # a second corridor with the same path: a tie
    g[8, 8] = 0                                                    # an isolated cell
    joint, ref = IncBinaryJoint(g.tolist()), IncBinary(g.tolist())
    edits = [(0, 3),      # cut the corridor that holds m: the untouched one (path 7) beats both halves
             (0, 3),      # mend it: path 7 in U and outside, the untouched component keeps m
             (4, 0),      # shorten the other one: no tie any more
             (8, 9),      # the isolated cell gets a neighbour (old isolated cell next to a cell that became passable)
             (8, 8),      # ... and goes, leaving the neighbour isolated (new isolated cell next to a solid cell)
             (8, 9),      # the last cell goes: an isolated cell became solid
             (12, 12),    # a new isolated cell
             (12, 13), (12, 14), (12, 13)]                         # grow it, then cut it into two isolated cells
    for y, x in edits:
        g[y, x] ^= 1
        ref.flip(y, x)
        joint.flip(y, x)
        _check(joint, g, (y, x))
        assert _state(joint) == _state(ref), (y, x)


def test_joint_update_on_narrow_rollouts():
    """Long narrow-representation rollouts on 16x16 maps, the flagship workload's edit pattern."""
    rng = np.random.default_rng(11)
    for _ in range(6):
        grid = rng.integers(0, 2, (16, 16)).astype(np.int64)
        joint, ref = IncBinaryJoint(grid.tolist()), IncBinary(grid.tolist())
        s0 = int(rng.integers(0, 256))
        for t in range(512):
            y, x = divmod((s0 + t) % 256, 16)
            v = int(rng.integers(0, 2))
            if v == grid[y, x]:
                continue
            grid[y, x] = v
            ref.flip(y, x)
            joint.flip(y, x)
            assert _state(joint) == _state(ref), (t, y, x)
        _check(joint, grid, "end")
