"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz by running the REAL reference.

Run in the build container (needs /root/reference):   python -m oracle.gen_golden
The fixtures are committed; the GPU box only ever reads the .npz files.

Two kinds of fixtures:
  stats_<problem>.npz    grids + the reference's own get_stats() output for each
  trace_<name>.npz       full episodes through the reference's real env stack
                         (PcgrlEnv + obs wrappers + ControlWrapper): per step action, reward,
                         done, stats, pos, grid (+ a few observations)
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import refshim as R  # noqa: E402
from oracle.pcgrl_oracle import STAT_NAMES, TILES  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

ZELDA_W = dict(player=3, key=3, door=3, regions=5, enemies=1, **{"nearest-enemy": 2, "path-length": 1})
BINARY_W = {"regions": 1, "path-length": 1}   # configs/task/binary.yaml


def ref_problem(problem, map_shape):
    R.install()
    from control_pcgrl.envs.probs import PROBLEMS
    cfg = R.make_cfg(problem, "narrow", map_shape, weights={})
    p = PROBLEMS[problem](cfg=cfg)
    p.adjust_param(cfg=cfg)
    return p


# (problem, map_shape) pairs of tests/golden/problem_tables.json
PROBLEM_TABLE_CASES = [("binary", (16, 16)), ("binary", (10, 14)), ("zelda", (7, 11)), ("zelda", (16, 16)),
                       ("sokoban", (5, 5)), ("sokoban", (6, 7)), ("smb", (116, 16)), ("minecraft_3D_maze", (14, 14, 14))]


def problem_table_key(problem, map_shape):
    return problem + "-" + "x".join(str(int(s)) for s in map_shape)


def problem_table(tiles, static_trgs, cond_bounds, reward_weights, border_tile):
    """What control_pcgrl_b200/problems.py restates of a Problem, in JSON form: the tile list, static targets and
    condition bounds as floats (a range target as a pair), the keys of the reward weights and the border tile."""
    def num(v):
        return [float(x) for x in v] if isinstance(v, (tuple, list)) else float(v)
    return {"tiles": [str(t) for t in tiles], "static_trgs": {k: num(v) for k, v in static_trgs.items()},
            "cond_bounds": {k: num(v) for k, v in cond_bounds.items()},
            "reward_weight_keys": sorted(reward_weights), "border_tile": str(border_tile)}


def problem_tables_fixture():
    """tests/golden/problem_tables.json: problem_table() of the reference's Problem classes for PROBLEM_TABLE_CASES.
    The committed file was written from control_pcgrl_b200/problems.py, because no reference tree was at hand when
    it was added; those tables had been compared with the real classes before, and the binary 16x16, zelda 7x11
    and minecraft 15^3 values agree with SURVEY.md section A (items 13-15).  Running this job with a reference tree
    rewrites it from the real classes."""
    import json
    out = {}
    for problem, shape in PROBLEM_TABLE_CASES:
        p = ref_problem(problem, shape)
        out[problem_table_key(problem, shape)] = problem_table(p.get_tile_types(), p.static_trgs, p.cond_bounds,
                                                               p._reward_weights, p._border_tile)
    with open(os.path.join(OUT, "problem_tables.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


def ref_stats(problem_obj, problem, grid):
    H = R.load_helpers()
    helper = H.h3 if grid.ndim == 3 else H.h2
    smap = helper.get_string_map(grid, TILES[problem])
    st = problem_obj.get_stats(smap)
    return [int(st[k]) for k in STAT_NAMES[problem]]


# ------------------------------------------------------------------------------------------ grids
def binary_grids():
    rng = np.random.default_rng(20261017)
    out = []
    for shape in [(16, 16)]:
        for p in (0.1, 0.2, 0.35, 0.5, 0.65, 0.8, 0.9):
            for _ in range(60):
                out.append((rng.random(shape) < p).astype(np.uint8))
    # hand-built known answers (SURVEY.md section C)
    out.append(np.zeros((16, 16), np.uint8))
    out.append(np.ones((16, 16), np.uint8))
    out.append((np.add.outer(np.arange(16), np.arange(16)) % 2).astype(np.uint8))
    serp = np.ones((16, 16), np.uint8)
    serp[0::2, :] = 0
    for i, y in enumerate(range(1, 16, 2)):
        serp[y, 15 if i % 2 == 0 else 0] = 0
    out.append(serp)
    rng2 = np.random.default_rng(12345)
    for _ in range(3):
        out.append((rng2.random((16, 16)) < 0.5).astype(np.uint8))
    return out


def binary_grids_other_shapes():
    rng = np.random.default_rng(7)
    out = []
    for shape in [(7, 11), (5, 5), (3, 20), (16, 18), (10, 14), (32, 32), (1, 1), (1, 9), (12, 1), (20, 27)]:
        for p in (0.2, 0.5, 0.7):
            for _ in range(8):
                out.append((rng.random(shape) < p).astype(np.uint8))
    R.install()
    from control_pcgrl.envs.probs.binary.eval_maps import binary_eval_maps
    out.append(np.array(binary_eval_maps[0]["map"], dtype=np.uint8))
    return out


def zelda_grids():
    rng = np.random.default_rng(99)
    out = []
    base = np.array([0.58, 0.3, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02])
    for shape in [(7, 11), (7, 11), (7, 11), (16, 16), (5, 9)]:
        for _ in range(60):
            out.append(rng.choice(8, size=shape, p=base).astype(np.uint8))
        # playable-ish: exactly one player/key/door planted on a sparse map
        for _ in range(60):
            g = rng.choice(8, size=shape, p=[0.7, 0.2, 0, 0, 0, 0.04, 0.03, 0.03]).astype(np.uint8)
            cells = rng.choice(g.size, size=3, replace=False)
            for c, t in zip(cells, (2, 3, 4)):
                g.flat[c] = t
            out.append(g)
    # reference level fixtures il/playable_maps/zelda_lvl*.txt (13x9 text incl. border; gen_trajectories.py:18-27)
    chars = {".": 0, "w": 1, "A": 2, "+": 3, "g": 4, "1": 5, "3": 6, "2": 7}
    d = os.path.join(R.REF_ROOT, "control_pcgrl", "il", "playable_maps")
    for i in range(50):
        with open(os.path.join(d, f"zelda_lvl{i}.txt")) as f:
            rows = [ln.rstrip("\n") for ln in f if ln.strip()]
        g = np.array([[chars[c] for c in r] for r in rows], dtype=np.uint8)[1:-1, 1:-1]
        out.append(g)
    return out


def sokoban_grids():
    rng = np.random.default_rng(31)
    out = []
    for shape in [(5, 5), (5, 5), (6, 7), (4, 8)]:
        for _ in range(60):
            out.append(rng.choice(5, size=shape, p=[0.45, 0.4, 0.05, 0.05, 0.05]).astype(np.uint8))
        # solver-friendly: one player, k crates, k targets, sparse walls (so _run_game actually runs)
        for _ in range(110):
            k = int(rng.integers(1, 4))
            g = (rng.random(shape) < rng.choice([0.0, 0.1, 0.2, 0.3])).astype(np.uint8)
            cells = rng.permutation(g.size)[:1 + 2 * k]
            g.flat[cells[0]] = 2
            g.flat[cells[1:1 + k]] = 3
            g.flat[cells[1 + k:]] = 4
            out.append(g)
    # harder: 7x7, 3-5 crates, open floor -- the BFS hits its 10 000-iteration cap and the A* passes decide
    for _ in range(40):
        k = int(rng.integers(3, 6))
        g = (rng.random((7, 7)) < rng.choice([0.05, 0.15])).astype(np.uint8)
        cells = rng.permutation(g.size)[:1 + 2 * k]
        g.flat[cells[0]] = 2
        g.flat[cells[1:1 + k]] = 3
        g.flat[cells[1 + k:]] = 4
        out.append(g)
    return out


def smb_grids():
    rng = np.random.default_rng(32)
    base = np.array([0.75, 0.1, 0.01, 0.04, 0.01, 0.02, 0.02])
    base /= base.sum()
    out = []
    for shape, n in [((116, 16), 50), ((16, 116), 24), ((16, 40), 30), ((12, 12), 40)]:
        for i in range(n):
            p = base
            if i % 4 == 3:
                p = rng.random(7)
                p /= p.sum()
            g = rng.choice(7, size=shape, p=p).astype(np.uint8)
            if i % 4 == 2:      # a solid ground row with gaps, like a real level
                g[-2:, :] = np.where(rng.random((2, shape[1])) < 0.85, 1, 0)
            out.append(g)
    return out


def floors_map(rng, size, wall_p=0.2, hole_p=0.15):
    """3D maps with storeys every 3 layers: long walks, stairs and jumps (random maps rarely have them)."""
    g = (rng.random((size,) * 3) < wall_p).astype(np.uint8)
    for z in range(3, size, 3):
        g[z] = (rng.random((size, size)) >= hole_p).astype(np.uint8)
    return g


def _test3d_maps():
    """The hand-built maps of the reference's test3D.py (test_map_1..23), read in place."""
    src = open(os.path.join(R.REF_ROOT, "test3D.py")).read().split("\n")
    start = next(i for i, ln in enumerate(src) if ln.startswith("test_map_1 "))
    end = next(i for i, ln in enumerate(src) if ln.startswith("def get_test_state"))
    ns = {}
    exec("\n".join(src[start:end]), ns)
    return [np.array(ns[f"test_map_{i}"]["map"], dtype=np.uint8) for i in range(1, 24)]


def maze3d_grids():
    rng = np.random.default_rng(33)
    out = []
    for size, n in [(14, 10), (10, 8), (8, 8), (6, 8)]:
        for p in (0.15, 0.3, 0.5, 0.7):
            for _ in range(n):
                out.append((rng.random((size,) * 3) < p).astype(np.uint8))
        for _ in range(n):
            out.append(floors_map(rng, size, wall_p=float(rng.choice([0.1, 0.2, 0.35])),
                                  hole_p=float(rng.choice([0.05, 0.15, 0.3]))))
    out.append(np.zeros((14, 14, 14), np.uint8))
    out.append(np.ones((14, 14, 14), np.uint8))
    H = R.load_helpers()
    kept = 0
    for m in _test3d_maps():
        try:        # non-cubic maps hit the IndexError of helper_3D.py:531 (SURVEY A-21)
            smap = H.h3.get_string_map(m, TILES["minecraft_3D_maze"])
            H.h3.calc_longest_path(smap, H.h3.get_tile_locations(smap, TILES["minecraft_3D_maze"]), ["AIR"])
        except IndexError:
            continue
        out.append(m)
        kept += 1
    print("test3D.py maps usable:", kept, "of 23")
    return out


def legacy_reward_fixture():
    """Random (new, old) stat pairs -> the reference's own Problem.get_reward (the non-ctrl classes)."""
    R.install()
    from control_pcgrl.envs.probs.binary.binary_prob import BinaryProblem
    from control_pcgrl.envs.probs.zelda.zelda_prob import ZeldaProblem
    from control_pcgrl.envs.probs.sokoban.sokoban_prob import SokobanProblem
    from control_pcgrl.envs.probs.smb.smb_prob import SMBProblem
    rng = np.random.default_rng(41)
    arrays = {}
    for problem, cls, shape, hi in [("binary", BinaryProblem, (16, 16), [130, 140]),
                                    ("zelda", ZeldaProblem, (7, 11), [3, 3, 12, 8, 6, 30, 60]),
                                    ("sokoban", SokobanProblem, (5, 5), [3, 6, 6, 4, 260, 30, 6]),
                                    ("smb", SMBProblem, (116, 16), [40, 8, 40, 1856, 60, 40, 30, 20, 60])]:
        cfg = R.make_cfg(problem, "narrow", shape, weights={})
        pobj = cls(cfg=cfg)
        names = STAT_NAMES[problem]
        new = np.stack([rng.integers(0, h + 1, size=400) for h in hi], axis=1)
        old = np.stack([rng.integers(0, h + 1, size=400) for h in hi], axis=1)
        if problem == "zelda":
            new[:, 6] -= 2
            old[:, 6] -= 2          # path-length can be -1 / -2
        if problem == "sokoban":
            new[:, 6] = np.abs(new[:, 1] - new[:, 2])
            old[:, 6] = np.abs(old[:, 1] - old[:, 2])
        out = []
        for a, b in zip(new, old):
            sn = {k: int(v) for k, v in zip(names, a)}
            so = {k: int(v) for k, v in zip(names, b)}
            if problem == "sokoban":
                sn["solution"] = [0] * sn["sol-length"]
                so["solution"] = [0] * so["sol-length"]
            out.append(float(pobj.get_reward(sn, so)))
        arrays[f"{problem}_new"], arrays[f"{problem}_old"], arrays[f"{problem}_reward"] = new, old, np.array(out)
    path = os.path.join(OUT, "legacy_reward.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path)


def save_stats_fixture(problem, grids, name=None):
    by_shape = {}
    for g in grids:
        by_shape.setdefault(g.shape, []).append(g)
    arrays = {}
    for i, (shape, gs) in enumerate(sorted(by_shape.items())):
        pobj = ref_problem(problem, shape)
        gs = np.stack(gs)
        st = np.array([ref_stats(pobj, problem, g) for g in gs], dtype=np.int64)
        arrays[f"grids_{i}"] = gs
        arrays[f"stats_{i}"] = st
    arrays["stat_names"] = np.array(STAT_NAMES[problem])
    path = os.path.join(OUT, f"stats_{name or problem}.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, {k: v.shape for k, v in arrays.items() if k.startswith("stats_")})


# ------------------------------------------------------------------------------------------ maps beyond 32x32
def binary_big_grids():
    """configs/task/binary_bigger.yaml:5 is 64x64: random maps at four densities, odd shapes with one side above
    32, the serpentine corridor (the longest possible path), all empty, all solid."""
    rng = np.random.default_rng(2024)
    bg = []
    for shape, n in (((64, 64), 10), ((40, 50), 8), ((33, 20), 6), ((17, 64), 6)):
        for k in range(n):
            bg.append((rng.random(shape) < (0.35, 0.5, 0.65, 0.8)[k % 4]).astype(np.uint8))
    g = np.ones((64, 64), np.uint8)
    for y in range(0, 64, 2):
        g[y, :] = 0
        g[y + 1 if y + 1 < 64 else y, 63 if (y // 2) % 2 == 0 else 0] = 0
    return bg + [g, np.zeros((64, 64), np.uint8), np.ones((64, 64), np.uint8)]


def zelda_big_grids():
    """configs/task/zelda_bigger.yaml:5 is 64x64: random levels, half of them with exactly one player / key / door so
    that both path searches run, a quarter mostly open (long reachable paths)."""
    rng = np.random.default_rng(2025)
    p = np.array([0.58, 0.3, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02])
    zg = []
    for shape, n in (((64, 64), 8), ((40, 50), 6), ((33, 20), 6)):
        for k in range(n):
            g = rng.choice(8, size=shape, p=p).astype(np.uint8)
            if k % 2 == 0:
                g[(g == 2) | (g == 3) | (g == 4)] = 0
                idx = rng.choice(g.size, 3, replace=False)
                g.flat[idx[0]], g.flat[idx[1]], g.flat[idx[2]] = 2, 3, 4
            if k % 4 == 0:
                g[(g == 1) & (rng.random(shape) < 0.7)] = 0
            zg.append(g)
    return zg


# ------------------------------------------------------------------------------------------ minecraft_2D_maze
def minecraft_2d_maze_fixture():
    """Minecraft2DmazeProblem.get_stats / get_reward (minecraft_2D_maze_prob.py:87-115), run verbatim.  The class
    cannot be constructed at this commit (its __init__ calls Problem.__init__() without the cfg it now requires,
    :15-16, and never sets the render_path its get_stats reads, :29), so the instance is made without __init__ and
    given the attributes those two methods read."""
    R.install()
    H = R.load_helpers()
    sys.modules["control_pcgrl.envs.probs.minecraft.mc_render"].spawn_2D_maze = lambda *a, **k: None
    sys.modules["control_pcgrl.envs.probs.minecraft.mc_render"].spawn_2D_path = lambda *a, **k: None
    sys.modules.setdefault("PIL", __import__("types").ModuleType("PIL")).Image = object
    from control_pcgrl.envs.probs.minecraft.minecraft_2D_maze_prob import Minecraft2DmazeProblem
    p = object.__new__(Minecraft2DmazeProblem)
    p.render_path = False
    p._reward_weights = {"regions": 5, "path-length": 1}
    rng = np.random.default_rng(77)
    arrays = {}
    for i, (shape, n, dens) in enumerate([((14, 14), 240, (0.2, 0.35, 0.5, 0.65, 0.8)), ((16, 16), 60, (0.5, 0.7)),
                                           ((9, 13), 60, (0.4, 0.6)), ((5, 5), 40, (0.5,))]):
        gs = np.stack([(rng.random(shape) < dens[k % len(dens)]).astype(np.int8) for k in range(n)])
        gs[0][:] = 0
        gs[1][:] = 1
        st = []
        for g in gs:
            smap = H.h2.get_string_map(g, ["AIR", "DIRT"])
            s = p.get_stats(smap)
            st.append([int(s["regions"]), int(s["path-length"])])
        arrays[f"grids_{i}"], arrays[f"stats_{i}"] = gs, np.array(st, dtype=np.int64)
    arrays["stat_names"] = np.array(STAT_NAMES["minecraft_2D_maze"])
    path = os.path.join(OUT, "stats_minecraft_2D_maze.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, {k: v.shape for k, v in arrays.items() if k.startswith("stats_")})
    new = np.stack([rng.integers(0, 60, size=300), rng.integers(0, 100, size=300)], axis=1)
    old = np.stack([rng.integers(0, 60, size=300), rng.integers(0, 100, size=300)], axis=1)
    rew = [float(p.get_reward(dict(zip(STAT_NAMES["minecraft_2D_maze"], a.tolist())),
                              dict(zip(STAT_NAMES["minecraft_2D_maze"], b.tolist())))) for a, b in zip(new, old)]
    path = os.path.join(OUT, "legacy_reward_minecraft_2D_maze.npz")
    np.savez_compressed(path, new=new, old=old, reward=np.array(rew))
    print("wrote", path)


# ------------------------------------------------------------------------------------------ holey problems
def ref_holey_problem(h, w):
    """The reference's BinaryHoleyProblem cannot be constructed at this commit (its __init__ calls
    BinaryProblem.__init__(self) without the cfg that now requires, binary_holey_prob.py:13-16, and
    PcgrlHoleyEnv.__init__ passes (prob, rep) where PcgrlCtrlEnv takes (cfg, prob, rep),
    pcgrl_holey_env.py:32-33), so the instance is made without running __init__ and given only the
    attributes its get_stats / hole helpers read.  get_stats, _valid_holes, get_border_idxs and
    gen_all_holes then run verbatim."""
    R.install()
    import sys as _sys
    _sys.modules["ray"].get = lambda x: x
    from control_pcgrl.envs.probs.binary.binary_holey_prob import BinaryHoleyProblem
    p = object.__new__(BinaryHoleyProblem)
    p._height, p._width = h, w
    p._tile_types = ["empty", "solid"]
    p._hole_queue, p.fixed_holes = [], False
    p._border_idxs = p.get_border_idxs()
    return p


def binary_holey_fixture():
    H = R.load_helpers()
    rng = np.random.default_rng(77)
    arrays = {}
    for gi, (h, w, n) in enumerate([(16, 16, 400), (10, 14, 120), (6, 6, 120), (30, 30, 40), (3, 5, 60)]):
        p = ref_holey_problem(h, w)
        border = p._border_idxs
        grids, holes, stats = [], [], []
        for i in range(n):
            dens = [0.1, 0.3, 0.45, 0.5, 0.55, 0.7, 0.9][i % 7]
            g = (rng.random((h, w)) < dens).astype(np.int8)
            if i % 11 == 0:
                g[:] = 0
            if i % 13 == 0:
                g[:] = 1
            if i % 17 == 0:   # a serpentine corridor: long entrance -> exit paths
                g[:] = 1
                for y in range(0, h, 2):
                    g[y, :] = 0
                    if y + 1 < h:
                        g[y + 1, (w - 1) if (y // 2) % 2 == 0 else 0] = 0
            if i % 5 == 0:    # the fixed holes of holey_prob.py:47-49
                e, x = np.array([1, 0]), np.array((w, h + 1))
                if x[0] > h + 1 or x[1] > w + 1:
                    k = rng.choice(len(border), 2, replace=False)
                    e, x = border[k[0]], border[k[1]]
            else:
                k = rng.choice(len(border), 2, replace=False)
                e, x = border[k[0]], border[k[1]]
            b = np.full((h + 2, w + 2), 1, dtype=np.int64)
            b[1:-1, 1:-1] = g
            b[e[0], e[1]] = 0
            b[x[0], x[1]] = 0
            p.entrance_coords, p.exit_coords = e, x
            st = p.get_stats(H.h2.get_string_map(b, ["empty", "solid"]))
            grids.append(g)
            holes.append([e[0], e[1], x[0], x[1]])
            stats.append([int(st[k2]) for k2 in STAT_NAMES["binary_holey"]])
        arrays[f"grids_{gi}"] = np.stack(grids)
        arrays[f"holes_{gi}"] = np.array(holes, dtype=np.int32)
        arrays[f"stats_{gi}"] = np.array(stats, dtype=np.int64)
        # _valid_holes / border order (pins the random-hole generator's validity rule)
        pairs = rng.choice(len(border), (200, 2))
        arrays[f"border_{gi}"] = border.astype(np.int32)
        arrays[f"valid_pairs_{gi}"] = pairs.astype(np.int32)
        arrays[f"valid_{gi}"] = np.array([bool(p._valid_holes(border[a], border[b2])) for a, b2 in pairs])
    arrays["stat_names"] = np.array(STAT_NAMES["binary_holey"])
    path = os.path.join(OUT, "stats_binary_holey.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, {k: v.shape for k, v in arrays.items() if k.startswith("stats_")})


def maze3d_holey_fixture():
    """minecraft_3D_holey_maze (oracle-only so far): sequences of get_stats calls on the reference's problem object
    (built without its broken constructor, like binary_holey), because `path-length` reports the de-stacked path
    of the PREVIOUS call.  Holes come from the reference's own gen_holes, cast to int64: its uint8 arrays make
    `x + dir` raise under numpy 2 (numpy 1 promoted to a wider int)."""
    R.install()
    import sys as _sys
    import types as _types
    _sys.modules["ray"].get = lambda x: x
    mr = _sys.modules["control_pcgrl.envs.probs.minecraft.mc_render"]
    setattr(mr, "spawn_3D_doors", lambda *a, **k: None)
    _sys.modules.setdefault("control_pcgrl.envs.probs.minecraft.minecraft_pb2",
                            _types.SimpleNamespace(BEDROCK=0, WOODEN_SLAB=0, LEAVES=0, TORCH=0, PURPUR_SLAB=0, WOOL=0))
    H = R.load_helpers()
    from control_pcgrl.envs.probs.minecraft.minecraft_3D_holey_maze_prob import Minecraft3DholeymazeProblem
    rng = np.random.default_rng(123)
    arrays = {}
    for gi, (size, trials, steps) in enumerate([(7, 60, 4), (10, 12, 3), (14, 5, 3)]):
        p = object.__new__(Minecraft3DholeymazeProblem)
        p._height = p._width = p._length = size
        p._tile_types = ["AIR", "DIRT"]
        p._hole_queue, p.fixed_holes = [], False
        p._border_idxs = p.get_border_idxs()
        maps, holes, stats = [], [], []
        for trial in range(trials):
            p.path_coords = []
            np.random.seed(1000 * gi + trial)
            if trial % 4 == 3:
                p.fixed_holes = True
            ent, ext = p.gen_holes()
            p.fixed_holes = False
            ent, ext = np.asarray(ent).astype(np.int64), np.asarray(ext).astype(np.int64)
            p.entrance_coords, p.exit_coords = ent, ext
            for step in range(steps):
                g = (rng.random((size,) * 3) < [0.2, 0.35, 0.5][trial % 3]).astype(np.int8)
                if trial % 5 == 0:
                    g[:] = 1
                    g[0:3] = 0            # an open hall on the floor
                if trial % 5 == 1:
                    g[:] = 1
                    g[0:2] = 0
                    g[2:5, :, ::3] = 0    # storeys reached by jumps / stairs
                b = np.ones((size + 2,) * 3, dtype=np.int8)
                b[1:-1, 1:-1, 1:-1] = g
                for hh in (ent, ext):
                    for c in hh:
                        b[c[0], c[1], c[2]] = 0
                st = p.get_stats(H.h3.get_string_map(b, ["AIR", "DIRT"]))
                maps.append(b)
                holes.append(np.stack([ent, ext]))
                stats.append([int(st[k]) for k in ("regions", "path-length", "connected-path-length", "n_jump")])
        arrays[f"maps_{gi}"] = np.stack(maps)
        arrays[f"holes_{gi}"] = np.stack(holes).astype(np.int32)
        arrays[f"stats_{gi}"] = np.array(stats, dtype=np.int64)
        arrays[f"steps_{gi}"] = np.array(steps)
    path = os.path.join(OUT, "stats_maze3d_holey.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, {k: v.shape for k, v in arrays.items() if k.startswith("stats_")})


def maze3d_holey_dungeon_fixture():
    """minecraft_3D_dungeon_holey: Minecraft3DholeyDungeonProblem.get_stats run verbatim on bordered maps with the
    holes dug (the instance is made without its constructor chain, broken upstream like the other holey problems)."""
    R.install()
    import sys as _sys
    import types as _types
    _sys.modules["ray"].get = lambda x: x
    mr = _sys.modules["control_pcgrl.envs.probs.minecraft.mc_render"]
    setattr(mr, "spawn_3D_doors", lambda *a, **k: None)
    _sys.modules.setdefault("control_pcgrl.envs.probs.minecraft.minecraft_pb2",
                            _types.SimpleNamespace(BEDROCK=0, WOODEN_SLAB=0, LEAVES=0, TORCH=0, PURPUR_SLAB=0, WOOL=0))
    if "sklearn.utils" not in _sys.modules or not hasattr(_sys.modules["sklearn.utils"], "check_X_y"):
        sk = _types.ModuleType("sklearn")
        sku = _types.ModuleType("sklearn.utils")
        sku.check_X_y = lambda *a, **k: None
        _sys.modules.setdefault("sklearn", sk)
        _sys.modules["sklearn.utils"] = sku
    H = R.load_helpers()
    from control_pcgrl.envs.probs.minecraft.minecraft_3D_holey_dungeon_prob import Minecraft3DholeyDungeonProblem
    TILES5 = ["AIR", "DIRT", "CHEST", "SKULL", "PUMPKIN"]
    rng = np.random.default_rng(321)
    arrays = {}
    for gi, (size, trials) in enumerate([(7, 120), (10, 40), (14, 16)]):
        p = object.__new__(Minecraft3DholeyDungeonProblem)
        p._height = p._width = p._length = size
        p._passable = set({"AIR", "CHEST", "SKULL", "PUMPKIN"})
        p._hole_queue, p.fixed_holes = [], False
        p._border_idxs = p.get_border_idxs()
        maps, holes, stats = [], [], []
        for trial in range(trials):
            np.random.seed(5000 * gi + trial)
            p.fixed_holes = trial % 4 == 3
            ent, ext = p.gen_holes()
            ent, ext = np.asarray(ent).astype(np.int64), np.asarray(ext).astype(np.int64)
            p.entrance_coords, p.exit_coords = ent, ext
            pr = [(0.55, 0.35, 0.04, 0.03, 0.03), (0.75, 0.2, 0.02, 0.02, 0.01), (0.5, 0.45, 0.0, 0.03, 0.02),
                  (0.6, 0.36, 0.04, 0.0, 0.0)][trial % 4]
            g = rng.choice(5, size=(size,) * 3, p=pr).astype(np.int8)
            if trial % 6 == 0:
                g[:] = 1
                g[0:3] = 0            # an open hall on the floor with a chest and enemies in it
                g[0, size // 2, size // 2] = 2
                g[0, 1, 1] = 3
                g[0, size - 2, 2] = 4
            b = np.ones((size + 2,) * 3, dtype=np.int8)
            b[1:-1, 1:-1, 1:-1] = g
            for hh in (ent, ext):
                for c in hh:
                    b[c[0], c[1], c[2]] = 0
            st = p.get_stats(H.h3.get_string_map(b, TILES5))
            maps.append(b)
            holes.append(np.stack([ent, ext]))
            stats.append([int(st[k]) for k in STAT_NAMES["minecraft_3D_dungeon_holey"]])
        arrays[f"maps_{gi}"] = np.stack(maps)
        arrays[f"holes_{gi}"] = np.stack(holes).astype(np.int32)
        arrays[f"stats_{gi}"] = np.array(stats, dtype=np.int64)
    arrays["stat_names"] = np.array(STAT_NAMES["minecraft_3D_dungeon_holey"])
    path = os.path.join(OUT, "stats_maze3d_holey_dungeon.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, {k: v.shape for k, v in arrays.items() if k.startswith("stats_")})


# ------------------------------------------------------------------------------------------ traces
def run_trace(name, problem, rep, map_shape, obs_window, weights, controls=None, n_envs=4, seed=0,
              max_board_scans=3, change_percentage=None, raw_only=False, n_steps=None, init_p=None,
              targets=None, obs_every=97, action_p=None, grid_every=1, act_window=None, static_prob=None):
    rng = np.random.default_rng(seed)
    cfg = R.make_cfg(problem, rep, map_shape, obs_window=obs_window, weights=weights, controls=controls,
                     max_board_scans=max_board_scans, change_percentage=change_percentage)
    # representation wrappers (envs/reps/wrappers.py wrap_rep :717-722)
    if act_window is not None:
        cfg.act_window = list(act_window)
    if static_prob is not None:
        cfg.static_tile_wrapper, cfg.static_prob = True, static_prob
    n_tiles = len(TILES[problem])
    rec = dict(grid0=[], pos0=[], actions=[], rewards=[], dones=[], stats=[], pos=[], grids=[], stats0=[],
               obs=[], obs_step=[], obs0=[], changes=[], trg=[], grids_step=[], static=[])
    for e in range(n_envs):
        env = R.make_wrapped_env(cfg, raw_only=raw_only)
        # every random draw of the reference itself (turtle start, frozen-tile mask and walls; the env's own
        # generator and the global numpy / python ones some wrappers use) is seeded, so a trace regenerates byte
        # for byte and a change of the generator cannot be mistaken for a change of the reference
        env.unwrapped.seed(100003 * seed + 17 * e + 1)
        np.random.seed(100003 * seed + 17 * e + 2)
        import random as _random
        _random.seed(100003 * seed + 17 * e + 3)
        if init_p is None:
            g0 = rng.integers(0, n_tiles, size=map_shape).astype(np.uint8)
        else:
            g0 = rng.choice(n_tiles, size=map_shape, p=init_p).astype(np.uint8)
        R.inject_map(env, g0)
        trg_e = []
        if targets is not None:
            t = {k: float(rng.uniform(*env.cond_bounds[k])) for k in targets}   # intended UniformNoiseyTargets
            env.set_trgs(t)
            trg_e = [t[k] for k in targets]
        ob, _ = env.reset()
        u = env.unwrapped
        rep_obj = u._rep.unwrapped
        static_e = np.zeros((0,), dtype=np.uint8)
        if static_prob is not None:
            w = u._rep
            while not hasattr(w, "static_tiles"):
                w = w.rep
            inner = tuple(slice(1, -1) for _ in map_shape)
            static_e = np.array(w.static_tiles[inner], dtype=np.uint8)      # interior of the bordered mask
        pos0 = [int(v) for v in rep_obj._pos] if rep in ("narrow", "turtle") else [0] * len(map_shape)
        stats0 = [int(u._rep_stats[k]) for k in STAT_NAMES[problem]]
        acts, rews, dones, stats, poss, grids, obs_l, obs_s, chg, grid_s = [], [], [], [], [], [], [], [], [], []
        done = False
        t = 0
        while not done and (n_steps is None or t < n_steps):
            if rep == "cellular":
                a = rng.random((n_tiles, *map_shape)).astype(np.float32)
                if t % 3 == 2:      # sometimes keep most of the map: near-no-op logits
                    a = np.moveaxis(np.eye(n_tiles, dtype=np.float32)[u._rep.unwrapped._map.astype(int)], -1, 0).copy()
                    if t % 6 == 2:
                        a[(slice(None), *[rng.integers(s) for s in map_shape])] = rng.random(n_tiles)
                act_store = a
            elif act_window is not None:
                a = rng.integers(0, n_tiles, size=int(np.prod(act_window)))
                if t % 4 == 3:      # sometimes a no-op patch (the current tiles) or a single-cell edit
                    tl = [int(rep_obj._pos[i]) - (act_window[i] - 1) // 2 for i in range(len(map_shape))]
                    cur = rep_obj._map[tuple(slice(tl[i], tl[i] + act_window[i]) for i in range(len(map_shape)))]
                    a = np.array(cur, dtype=np.int64).reshape(-1)
                    if t % 8 == 7:
                        a[rng.integers(a.size)] = rng.integers(n_tiles)
                act_store = np.array(a)
            elif rep == "wide" and raw_only:
                a = [int(rng.integers(s)) for s in map_shape] + [int(rng.integers(n_tiles))]
                act_store = np.array(a)
            else:
                a = int(rng.integers(env.action_space.n)) if action_p is None else \
                    int(rng.choice(env.action_space.n, p=action_p))
                act_store = a
            ob, r, done, trunc, info = env.step(a)
            acts.append(act_store)
            rews.append(float(r))
            dones.append(bool(done))
            stats.append([int(u._rep_stats[k]) for k in STAT_NAMES[problem]])
            p = getattr(rep_obj, "_pos", None)
            poss.append([int(v) for v in p] if p is not None and rep in ("narrow", "turtle") else [0] * len(map_shape))
            chg.append(int(info["changes"]))
            if t % grid_every == 0 or done or (n_steps is not None and t + 1 == n_steps):
                grids.append(np.array(rep_obj._map, dtype=np.uint8))
                grid_s.append(t)
            if (t % obs_every == 0 or done) and not raw_only:
                obs_l.append(np.asarray(ob, dtype=np.float64))
                obs_s.append(t)
            t += 1
        rec["grid0"].append(g0); rec["pos0"].append(pos0); rec["stats0"].append(stats0)
        rec["actions"].append(np.array(acts)); rec["rewards"].append(rews); rec["dones"].append(dones)
        rec["stats"].append(stats); rec["pos"].append(poss); rec["grids"].append(np.stack(grids))
        rec["obs"].append(np.stack(obs_l) if obs_l else np.zeros((0,))); rec["obs_step"].append(obs_s)
        rec["changes"].append(chg); rec["trg"].append(trg_e); rec["grids_step"].append(grid_s)
        rec["static"].append(static_e)
    arrays = {"n_envs": np.array(n_envs)}
    for k, v in rec.items():
        if k == "obs0":
            continue
        for e in range(n_envs):          # episodes can be ragged (change_percentage) -> one array per env
            arrays[f"{k}_{e}"] = np.array(v[e])
    arrays["meta_problem"] = np.array(problem); arrays["meta_rep"] = np.array(rep)
    arrays["meta_map_shape"] = np.array(map_shape); arrays["meta_obs_window"] = np.array(obs_window)
    arrays["meta_max_board_scans"] = np.array(max_board_scans)
    arrays["meta_change_percentage"] = np.array(-1.0 if change_percentage is None else change_percentage)
    arrays["meta_controls"] = np.array(controls or [], dtype=str)
    arrays["meta_weight_keys"] = np.array(list(weights.keys()), dtype=str)
    arrays["meta_weight_vals"] = np.array(list(weights.values()), dtype=np.float64)
    arrays["meta_raw_only"] = np.array(raw_only)
    arrays["meta_targets"] = np.array(targets or [], dtype=str)
    arrays["meta_act_window"] = np.array(act_window or [], dtype=np.int64)
    arrays["meta_static"] = np.array(static_prob is not None)
    path = os.path.join(OUT, f"trace_{name}.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, "steps", [arrays[f"rewards_{e}"].shape[0] for e in range(n_envs)], "bytes", os.path.getsize(path))


def multiagent_fixture():
    """Multi-agent turtle through the reference's real stack: CroppedImagePCGRLWrapper + ControlWrapper +
    MultiAgentWrapper (rl/envs.py:28-76, wrappers.py:697-736) over MultiAgentTurtleRepresentation
    (envs/reps/wrappers.py:612-651).  One multi-agent step is one full env step per agent, in dict order; every
    agent's observation is taken right after its own sub-step.  -> tests/golden/multiagent_turtle.npz"""
    import random as _random
    from types import SimpleNamespace
    R.install()
    from control_pcgrl import wrappers
    ZP = [0.58, 0.3, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02]
    # last field: cfg.show_agents (ShowAgentRepresentation, envs/reps/wrappers.py:189-232: an 'agent_occupancy' plane)
    cases = [("binary", (8, 8), (16, 16), BINARY_W, 2, None, None, 3, False),
             ("zelda", (7, 11), (22, 22), ZELDA_W, 3, ZP, None, 2, False),
             ("binary", (10, 6), (20, 20), BINARY_W, 4, None, 0.3, 2, False),
             ("zelda", (7, 11), (10, 12), ZELDA_W, 3, ZP, None, 2, True)]
    arrays = {"n_cases": np.array(len(cases))}
    for ci, (problem, map_shape, obs_window, weights, n_agents, init_p, chg_pct, n_envs, show) in enumerate(cases):
        rng = np.random.default_rng(900 + ci)
        cfg = R.make_cfg(problem, "turtle", map_shape, obs_window=obs_window, weights=weights,
                         change_percentage=chg_pct)
        cfg.multiagent = SimpleNamespace(n_agents=n_agents)
        cfg.show_agents = show
        arrays[f"c{ci}_show_agents"] = np.array(show)
        n_tiles = len(TILES[problem])
        arrays[f"c{ci}_problem"] = np.array(problem)
        arrays[f"c{ci}_map_shape"] = np.array(map_shape)
        arrays[f"c{ci}_obs_window"] = np.array(obs_window)
        arrays[f"c{ci}_n_agents"] = np.array(n_agents)
        arrays[f"c{ci}_n_envs"] = np.array(n_envs)
        arrays[f"c{ci}_change_percentage"] = np.array(-1.0 if chg_pct is None else chg_pct)
        arrays[f"c{ci}_weight_keys"] = np.array(list(weights.keys()), dtype=str)
        arrays[f"c{ci}_weight_vals"] = np.array(list(weights.values()), dtype=np.float64)
        for e in range(n_envs):
            env = R.make_wrapped_env(cfg)
            menv = wrappers.MultiAgentWrapper(env, cfg)
            env.unwrapped.seed(7000 + 31 * ci + e)
            np.random.seed(7100 + 31 * ci + e)
            _random.seed(7200 + 31 * ci + e)
            g0 = (rng.integers(0, n_tiles, size=map_shape) if init_p is None else
                  rng.choice(n_tiles, size=map_shape, p=init_p)).astype(np.uint8)
            R.inject_map(env, g0)
            obs, _ = menv.reset()
            u = env.unwrapped
            rep = u._rep
            names = [f"agent_{i}" for i in range(n_agents)]
            pos0 = np.array(rep.agent_positions, dtype=np.int64).copy()
            obs0 = np.stack([np.asarray(obs[k], dtype=np.float64) for k in names])
            stats0 = [int(u._rep_stats[k]) for k in STAT_NAMES[problem]]
            acts, rews, dones, stats, poss, grids, obs_l, obs_s, its, chg = [], [], [], [], [], [], [], [], [], []
            t, all_done = 0, False
            while not all_done and t < 600:
                a = {k: int(rng.integers(env.action_space.n)) for k in names}
                # the wrapper steps the agents one after the other; the per-agent stats / positions are read by
                # doing the same loop here (wrappers.py:724-731)
                st_t, pos_t, rew_t, done_t, ob_t = [], [], [], [], []
                for k in names:
                    u._rep.set_active_agent(k)
                    ob_k, r_k, d_k, tr_k, info_k = env.step({k: a[k]})
                    st_t.append([int(u._rep_stats[m]) for m in STAT_NAMES[problem]])
                    pos_t.append(np.array(rep.agent_positions, dtype=np.int64).copy())
                    rew_t.append(float(r_k))
                    done_t.append(bool(d_k))
                    ob_t.append(np.asarray(ob_k[k], dtype=np.float64))
                acts.append([a[k] for k in names]); rews.append(rew_t); dones.append(done_t); stats.append(st_t)
                poss.append(pos_t)
                its.append(int(info_k["iterations"])); chg.append(int(info_k["changes"]))
                grids.append(np.array(rep.unwrapped._map, dtype=np.uint8))
                if t % 37 == 0:
                    obs_l.append(np.stack(ob_t)); obs_s.append(t)
                all_done = all(done_t)
                t += 1
            pre = f"c{ci}_e{e}_"
            arrays[pre + "grid0"] = g0; arrays[pre + "pos0"] = pos0; arrays[pre + "obs0"] = obs0
            arrays[pre + "stats0"] = np.array(stats0)
            arrays[pre + "actions"] = np.array(acts); arrays[pre + "rewards"] = np.array(rews)
            arrays[pre + "dones"] = np.array(dones); arrays[pre + "stats"] = np.array(stats)
            arrays[pre + "pos"] = np.array(poss); arrays[pre + "grids"] = np.stack(grids)
            arrays[pre + "obs"] = np.stack(obs_l); arrays[pre + "obs_step"] = np.array(obs_s)
            arrays[pre + "iterations"] = np.array(its); arrays[pre + "changes"] = np.array(chg)
            print("multiagent", problem, map_shape, "agents", n_agents, "env", e, "steps", t)
    path = os.path.join(OUT, "multiagent_turtle.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, "bytes", os.path.getsize(path))


def main(which=None):
    os.makedirs(OUT, exist_ok=True)
    jobs = {
        "stats_binary": lambda: save_stats_fixture("binary", binary_grids()),
        "stats_binary_shapes": lambda: save_stats_fixture("binary", binary_grids_other_shapes(), "binary_shapes"),
        "stats_zelda": lambda: save_stats_fixture("zelda", zelda_grids()),
        "trace_binary_narrow": lambda: run_trace("binary_narrow", "binary", "narrow", (16, 16), (32, 32), BINARY_W),
        "trace_binary_narrow_chg": lambda: run_trace("binary_narrow_chg", "binary", "narrow", (16, 16), (32, 32),
                                                     BINARY_W, change_percentage=0.2, seed=1),
        "trace_binary_turtle": lambda: run_trace("binary_turtle", "binary", "turtle", (16, 16), (32, 32), BINARY_W, seed=2),
        "trace_binary_wide_ctrl": lambda: run_trace("binary_wide_ctrl", "binary", "wide", (16, 16), (16, 16), BINARY_W,
                                                    controls=["regions", "path-length"], seed=3,
                                                    targets=["regions", "path-length"]),
        "trace_binary_cellular": lambda: run_trace("binary_cellular", "binary", "cellular", (16, 16), (16, 16), BINARY_W,
                                                   seed=4, raw_only=True, n_steps=40, n_envs=2),
        "trace_zelda_turtle": lambda: run_trace("zelda_turtle", "zelda", "turtle", (7, 11), (22, 22), ZELDA_W, seed=5,
                                                init_p=[0.58, 0.3, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02], obs_every=61),
        "trace_zelda_narrow": lambda: run_trace("zelda_narrow", "zelda", "narrow", (7, 11), (22, 22), ZELDA_W, seed=6,
                                                init_p=[0.58, 0.3, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02], obs_every=61),
        "trace_zelda_wide_raw": lambda: run_trace("zelda_wide_raw", "zelda", "wide", (7, 11), (7, 11), ZELDA_W, seed=7,
                                                  raw_only=True, n_envs=2,
                                                  init_p=[0.58, 0.3, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02]),
    }
    SOK_W = {"player": 3, "crate": 2, "regions": 5, "ratio": 2, "dist-win": 0.5, "sol-length": 1}
    SMB_W = {"dist-floor": 2, "disjoint-tubes": 1, "enemies": 1, "empty": 1, "noise": 4, "jumps": 2,
             "jumps-dist": 2, "dist-win": 5, "sol-length": 1}
    MC_W = {"regions": 1, "path-length": 2, "n_jump": 3}
    SOK_P = [0.45, 0.4, 0.05, 0.05, 0.05]
    SOK_AP = [0.62, 0.12, 0.04, 0.11, 0.11]        # biased so the solver preconditions hold now and then
    SMB_P = list(np.array([0.75, 0.1, 0.01, 0.04, 0.01, 0.02, 0.02]) / 0.95)
    jobs.update({
        "legacy_reward": legacy_reward_fixture,
        "multiagent_turtle": multiagent_fixture,
        "stats_sokoban": lambda: save_stats_fixture("sokoban", sokoban_grids()),
        "stats_smb": lambda: save_stats_fixture("smb", smb_grids()),
        "stats_maze3d": lambda: save_stats_fixture("minecraft_3D_maze", maze3d_grids(), "maze3d"),
        "trace_sokoban_narrow": lambda: run_trace("sokoban_narrow", "sokoban", "narrow", (5, 5), (10, 10), SOK_W, seed=11,
                                                  init_p=SOK_AP, action_p=SOK_AP, n_envs=6, obs_every=17),
        "trace_sokoban_turtle": lambda: run_trace("sokoban_turtle", "sokoban", "turtle", (5, 5), (10, 10), SOK_W, seed=12,
                                                  init_p=SOK_AP, n_envs=4, obs_every=17),
        "trace_sokoban_cellular": lambda: run_trace("sokoban_cellular", "sokoban", "cellular", (5, 5), (5, 5), SOK_W,
                                                    seed=13, raw_only=True, n_envs=3, init_p=SOK_P),
        "trace_smb_narrow": lambda: run_trace("smb_narrow", "smb", "narrow", (116, 16), (32, 32), SMB_W, seed=14,
                                              init_p=SMB_P, n_envs=2, n_steps=300, grid_every=100, obs_every=233),
        "trace_smb_narrow_small": lambda: run_trace("smb_narrow_small", "smb", "narrow", (20, 16), (32, 32), SMB_W,
                                                    seed=20, init_p=SMB_P, n_envs=2, grid_every=60, obs_every=233),
        "trace_smb_turtle_small": lambda: run_trace("smb_turtle_small", "smb", "turtle", (14, 20), (28, 28), SMB_W,
                                                    seed=15, init_p=SMB_P, n_envs=2, grid_every=50, obs_every=211),
        "trace_maze3d_narrow": lambda: run_trace("maze3d_narrow", "minecraft_3D_maze", "narrow", (14, 14, 14),
                                                 (14, 14, 14), MC_W, seed=16, raw_only=True, n_envs=2, n_steps=400,
                                                 grid_every=100),
        "trace_maze3d_turtle": lambda: run_trace("maze3d_turtle", "minecraft_3D_maze", "turtle", (7, 7, 7), (7, 7, 7),
                                                 MC_W, seed=17, raw_only=True, n_envs=2, grid_every=50),
        "trace_maze3d_wide_raw": lambda: run_trace("maze3d_wide_raw", "minecraft_3D_maze", "wide", (6, 6, 6), (6, 6, 6),
                                                   MC_W, seed=18, raw_only=True, n_envs=2, grid_every=40),
        "trace_maze3d_cellular": lambda: run_trace("maze3d_cellular", "minecraft_3D_maze", "cellular", (6, 6, 6),
                                                   (6, 6, 6), MC_W, seed=19, raw_only=True, n_envs=2, n_steps=30,
                                                   init_p=[0.5, 0.5]),
    })
    # representation wrappers: MultiActionRepresentation (narrow only upstream) and StaticTileRepresentation
    # (narrow / turtle only upstream)
    ZP = [0.58, 0.3, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02]
    jobs.update({
        "trace_binary_patch33": lambda: run_trace("binary_patch33", "binary", "narrow", (16, 16), (32, 32), BINARY_W,
                                                  seed=30, act_window=(3, 3), n_envs=3, max_board_scans=1, grid_every=7),
        "trace_binary_patch42_chg": lambda: run_trace("binary_patch42_chg", "binary", "narrow", (16, 16), (32, 32),
                                                      BINARY_W, seed=31, act_window=(4, 2), n_envs=3,
                                                      change_percentage=0.4, grid_every=7),
        "trace_zelda_squeegee": lambda: run_trace("zelda_squeegee", "zelda", "narrow", (7, 11), (22, 22), ZELDA_W,
                                                  seed=32, act_window=(7, 1), n_envs=2, init_p=ZP, grid_every=3),
        "trace_maze3d_patch": lambda: run_trace("maze3d_patch", "minecraft_3D_maze", "narrow", (6, 6, 6), (6, 6, 6), MC_W,
                                                seed=33, raw_only=True, n_envs=2, act_window=(2, 3, 2), grid_every=20,
                                                init_p=[0.5, 0.5]),
        "trace_binary_static_narrow": lambda: run_trace("binary_static_narrow", "binary", "narrow", (16, 16), (32, 32),
                                                        BINARY_W, seed=34, static_prob=0.8, n_envs=4, grid_every=11,
                                                        change_percentage=0.5),
        "trace_zelda_static_turtle": lambda: run_trace("zelda_static_turtle", "zelda", "turtle", (7, 11), (22, 22),
                                                       ZELDA_W, seed=35, static_prob=0.9, n_envs=3, init_p=ZP,
                                                       grid_every=5, obs_every=31),
        "trace_binary_static_patch": lambda: run_trace("binary_static_patch", "binary", "narrow", (16, 16), (32, 32),
                                                       BINARY_W, seed=36, static_prob=0.7, act_window=(3, 3), n_envs=3,
                                                       max_board_scans=1, grid_every=7),
        "trace_sokoban_static_narrow": lambda: run_trace("sokoban_static_narrow", "sokoban", "narrow", (5, 5), (10, 10),
                                                         SOK_W, seed=37, static_prob=0.6, init_p=SOK_AP, action_p=SOK_AP,
                                                         n_envs=3, obs_every=17),
    })
    jobs["stats_binary_big"] = lambda: save_stats_fixture("binary", binary_big_grids(), "binary_big")
    jobs["stats_zelda_big"] = lambda: save_stats_fixture("zelda", zelda_big_grids(), "zelda_big")
    jobs["stats_binary_holey"] = binary_holey_fixture
    jobs["stats_minecraft_2D_maze"] = minecraft_2d_maze_fixture
    jobs["stats_maze3d_holey"] = maze3d_holey_fixture
    jobs["stats_maze3d_holey_dungeon"] = maze3d_holey_dungeon_fixture
    jobs["problem_tables"] = problem_tables_fixture
    for k, fn in jobs.items():
        if which and k not in which:
            continue
        fn()


if __name__ == "__main__":
    main(sys.argv[1:] or None)
