"""GPU: the skipped final sweep of BinaryIncMachine at its boundary, on hand-built 16x16 maps.

When an edit does not touch the component that held the maximum, the machine skips the final sweep if the first
sweeps bound every far tile's eccentricity in U by path-length (tests/inc_oracle_skip.py).  The edits below bring
that bound exactly to path-length (skipped; on the tie m stays in the old component) and one above it with an
eccentricity one above path-length (swept, path-length and m move), then keep editing, so that a wrong m or a wrong
far tile would surface in later stats.  The three-launch (`inc`) and one-launch (`incfused`) paths run the machine;
the lane-group kernel (`lg`) runs its own restatement without the skip and serves as the reference for the cache
rows.  Every step is checked against stats computed from scratch."""
import numpy as np
import pytest
import torch

from tests.inc_oracle_skip import IncBinarySkip

pytestmark = pytest.mark.gpu

PATHS = ["inc", "incfused", "lg"]

# (y, x, whether the CPU restatement skips the final sweep, path-length after the edit)
EDITS = [
    # a straight corridor in row 12 grows from its first tile (12, 0): e1 = lu = its length - 1
    *[(12, x, 2 * x <= 8, 8) for x in range(9)],   # skipped while 2 * e1 <= 8 = path, then swept; the last one ties
    (8, 2, True, 8),       # the U's left arm: e1 = 4, 2 * e1 = lu = path: skipped, a tie (m stays in row 0)
    (12, 9, False, 9),     # the row-12 corridor: lu = path + 1: swept, path and m move
    (12, 9, False, 8),     # shorten it again: the component of m is edited, joint sweep, three-way tie
    (9, 2, False, 9),      # the U's left arm: e1 = 5, 2 * e1 = 10 > path, lu = 9 = path + 1: path and m move
    (0, 4, True, 9),       # cut the row-0 corridor: halves with e1 = 3 and 4
    (12, 3, True, 9),      # cut the row-12 corridor: halves with e1 = 2 and 4
    (4, 3, False, 5),      # cut the U at its top bar (m's component): its left arm is left, path 5
    (0, 4, False, 8),      # mend the row-0 corridor: lu = 8 > 5
    (12, 3, False, 8),     # mend the row-12 corridor: swept (2 * e1 = 16), a tie: m stays
    (12, 0, False, 8),     # the row-12 corridor loses its first tile
    (12, 9, False, 8),     # ... and grows at the other end: a tie again
    (12, 10, False, 9),    # lu = 9 from the new first tile (12, 1)
]


def _map():
    g = np.ones((16, 16), dtype=np.int8)
    g[0, 0:9] = 0          # a corridor of path 8: holds path-length and m
    g[4, 2:5] = 0          # an upside-down U whose first tile is its corner (4, 2): top bar of 3 cells,
    g[5:8, 2] = 0          # left arm of 3 cells below the corner (4 with (8, 2), 5 with (9, 2)),
    g[5:7, 4] = 0          # right arm of 2 cells: the far tile of the corner lies at depth 4
    return g


def test_skip_boundary_on_hand_built_maps(monkeypatch):
    import control_pcgrl_b200 as P
    cfg = P.make_config("binary", "wide", map_shape=(16, 16), obs_window=(16, 16))
    envs = [P.BatchedPcgrlEnv(cfg, 1, action_kind="wide_coords") for _ in PATHS]
    g = _map()
    cpu = IncBinarySkip(g.tolist())
    assert cpu.path == 8
    for e in envs:
        e.reset(grids=g[None])
    for step, (y, x, skipped, path) in enumerate(EDITS):
        g[y, x] ^= 1
        before = cpu.skipped
        cpu.flip(y, x)
        assert (cpu.skipped > before, cpu.path) == (skipped, path), (step, y, x)
        a = torch.tensor([[y, x, int(g[y, x])]], dtype=torch.int32, device=envs[0].device)
        for path_name, e in zip(PATHS, envs):
            monkeypatch.setenv("PCGRL_STEP_PATH", path_name)
            e.step(a)
            assert np.array_equal(e.maps[0].cpu().numpy(), g), (step, path_name)
            fresh = e.compute_stats(e.maps)
            assert torch.equal(fresh, e.stats), (step, path_name, fresh.tolist(), e.stats.tolist())
            assert e.stats[0].tolist() == [cpu.regions, cpu.path], (step, path_name)
        assert torch.equal(envs[0].cache, envs[2].cache), step
        assert torch.equal(envs[1].cache, envs[2].cache), step
    for e in envs:
        e.check_status()
