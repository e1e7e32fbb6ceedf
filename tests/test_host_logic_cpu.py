"""CPU: host-side logic -- registry ids, config normalisation, problem tables, sharding, gloo reduction."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import control_pcgrl_b200 as P
from control_pcgrl_b200 import config as C
from control_pcgrl_b200 import problems, registry
from control_pcgrl_b200.dist import shard_range

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_registry_ids_follow_the_reference_scheme():
    # control_pcgrl/__init__.py:26-30: '{prob}-{rep}-v0' for every pair; plus the stale 3D spellings
    for prob in ("binary", "zelda", "sokoban", "smb", "minecraft_3D_maze"):
        for rep in ("narrow", "turtle", "wide", "cellular"):
            assert registry.parse_id(f"{prob}-{rep}-v0") == {"prob": prob, "rep": rep}
    assert registry.parse_id("minecraft_3D_maze-narrow3D-v0")["rep"] == "narrow"
    with pytest.raises(KeyError):
        registry.parse_id("nope-narrow-v0")


def test_config_normalise_accepts_all_flavours():
    from types import SimpleNamespace
    d = C.make_config("zelda", "turtle")
    n = C.normalise(d)
    assert n.map_shape == (7, 11) and n.obs_window == (22, 22) and n.weights["regions"] == 5
    ns = SimpleNamespace(task=SimpleNamespace(problem="binary", map_shape=[16, 16], obs_window=[32, 32], weights={}),
                         representation="narrow", max_board_scans=3, change_percentage=None, controls=None)
    assert C.normalise(ns).map_shape == (16, 16)
    dd = {"task": {"problem": "binary", "map_shape": (16, 16), "obs_window": (16, 16), "weights": {}},
          "representation": "wide", "controls": ["regions"]}
    assert C.normalise(dd).controls == ["regions"]
    assert d.env_name == "zelda-turtle-v0"


def test_problem_tables_known_constants():
    # SURVEY.md A-13 / A-14
    b = problems.get_spec("binary", (16, 16))
    assert b.static_trgs == {"regions": 1, "path-length": 136.0}
    assert b.cond_bounds == {"regions": (0, 128.0), "path-length": (0, 136.0)}
    z = problems.get_spec("zelda", (7, 11))
    assert z.static_trgs["path-length"] == 89 and z.static_trgs["nearest-enemy"] == (5, 49)
    assert z.cond_bounds["regions"] == (0, 38.5) and z.cond_bounds["player"] == (0, 75)


@pytest.mark.parametrize("problem,shape", [("binary", (16, 16)), ("binary", (10, 14)), ("zelda", (7, 11)),
                                           ("zelda", (16, 16)), ("sokoban", (5, 5)), ("sokoban", (6, 7)),
                                           ("smb", (116, 16)), ("minecraft_3D_maze", (14, 14, 14))])
def test_problem_tables_match_reference_classes(problem, shape):
    """The problem tables against the reference's Problem classes: their values recorded in
    tests/golden/problem_tables.json (oracle/gen_golden.py), and the live classes too when a reference tree exists."""
    from oracle import refshim as R
    from oracle.gen_golden import problem_table, problem_table_key, ref_problem
    with open(os.path.join(ROOT, "tests", "golden", "problem_tables.json")) as f:
        want = json.load(f)[problem_table_key(problem, shape)]
    spec = problems.get_spec(problem, shape)
    assert problem_table(spec.tiles, spec.static_trgs, spec.cond_bounds, spec.reward_weights, spec.border_tile) == want
    if R.available():
        ref = ref_problem(problem, shape)
        assert problem_table(ref.get_tile_types(), ref.static_trgs, ref.cond_bounds, ref._reward_weights,
                             ref._border_tile) == want


@pytest.mark.needs_reference
@pytest.mark.parametrize("mod,cls", [("microstructure.microstructure_prob", "MicroStructureProblem"),
                                     ("ddave.ddave_prob", "DDaveProblem"), ("mdungeon.mdungeon_prob", "MDungeonProblem"),
                                     ("loderunner_prob", "LoderunnerProblem"),
                                     ("loderunner_ctrl_prob", "LoderunnerCtrlProblem")])
def test_unbuilt_rank4_problems_are_dead_upstream(mod, cls):
    """DESIGN.md section 9: the helper-based problems that are NOT built cannot be constructed in the reference at
    this commit -- `__init__(self)` calls `super().__init__()` while Problem.__init__ needs the config."""
    import importlib
    from oracle import refshim as R
    R.install()
    C = getattr(importlib.import_module("control_pcgrl.envs.probs." + mod), cls)
    with pytest.raises(TypeError):
        C(cfg=R.make_cfg("binary", "narrow", (8, 8)))
    with pytest.raises(TypeError):
        C()


def test_shard_range_partitions_exactly():
    for n in (0, 1, 7, 65536, 1000003):
        for w in (1, 2, 3, 8):
            rngs = [shard_range(n, r, w) for r in range(w)]
            assert rngs[0][0] == 0 and rngs[-1][1] == n
            assert all(rngs[i][1] == rngs[i + 1][0] for i in range(w - 1))
            sizes = [b - a for a, b in rngs]
            assert max(sizes) - min(sizes) <= 1


GLOO_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
from control_pcgrl_b200.dist import init_from_env, reduce_episode_stats, shard_range
rank, local, world = init_from_env("gloo")
lo, hi = shard_range(1000, rank, world)
g = torch.Generator().manual_seed(123)
allv = torch.randint(0, 137, (1000, 3), generator=g).double()
out = reduce_episode_stats(allv[lo:hi], names=["a", "b", "c"])
assert out["count"] == 1000
assert torch.allclose(out["mean"], allv.mean(0)), (out["mean"], allv.mean(0))
assert torch.allclose(out["std"], allv.std(0, unbiased=False))
assert torch.equal(out["max"], allv.max(0).values) and torch.equal(out["min"], allv.min(0).values)
# an empty shard must not poison the reduction
out2 = reduce_episode_stats(allv[lo:hi] if rank == 0 else allv[:0])
assert out2["count"] == hi - lo if rank == 0 else True
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_episode_stat_reduction_gloo_world2(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(GLOO_WORKER.format(root=ROOT))
    port = 29500 + (os.getpid() % 400)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=180)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("ok" in o for o in outs)


def test_bench_reference_arm_prints_contract_line():
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "5",
                                   "--warmup", "1"], text=True, timeout=300)
    import json
    line = json.loads(out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "env-steps/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["config"]["workload"] == "binary-narrow-16x16"
