#!/usr/bin/env python
"""Small invocations of every kernel family, for `compute-sanitizer --tool memcheck python scripts/memcheck_small.py`."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import control_pcgrl_b200 as P  # noqa: E402


def roll(problem, rep, shape, n, steps, path=None, **kw):
    if path:
        os.environ["PCGRL_STEP_PATH"] = path
    cfg_kw = {k: v for k, v in kw.items() if k in ("controls", "obs_window", "act_window", "fixed_holes")}
    env = P.BatchedPcgrlEnv(P.make_config(problem, rep, map_shape=shape, max_board_scans=0.05, **cfg_kw), n, seed=1,
                            auto_reset=True, action_kind=kw.get("action_kind"), compact_host_io=kw.get("compact", False))
    env.reset()
    n_act = env.n_tiles + (4 if rep == "turtle" else 0)
    g = torch.Generator(device=env.device).manual_seed(0)
    for t in range(steps):
        if rep == "cellular":
            a = torch.randint(0, env.n_tiles, (n, env.row_stride), generator=g, device=env.device).to(torch.int8)
            a[:, env.cells:] = 0
        elif rep == "wide":
            a = torch.randint(0, shape[0] * shape[1] * env.n_tiles, (n,), generator=g, device=env.device, dtype=torch.int32)
        else:
            a = torch.randint(0, n_act, (n,), generator=g, device=env.device, dtype=torch.int32)
        if kw.get("compact"):
            env.step_host(a.cpu().numpy())
        else:
            env.step(a)
    if not env.ctrl_metrics:          # target planes are fractional: float observations only
        env.observe(dtype=torch.uint8)
        env.observe(dtype=torch.uint8, onehot=False)
    env.observe(dtype=torch.float32)
    torch.cuda.synchronize()
    env.check_status()
    os.environ.pop("PCGRL_STEP_PATH", None)
    print("ok", problem, rep, shape, path or "", flush=True)


# the kernels added last (lane groups).  MEMCHECK_ONLY=new stops after them.
for shape, rep in (((16, 16), "narrow"), ((7, 5), "turtle"), ((3, 4), "narrow"), ((2, 16), "narrow")):
    roll("binary", rep, shape, 3000, 40, "lg")
roll("binary", "narrow", (16, 16), 50000, 12, "lg")            # 16 envs per warp
if os.environ.get("MEMCHECK_ONLY") == "new":
    sys.exit(0)
for path in ("fused", "split", "inc", "incfused"):
    roll("binary", "narrow", (16, 16), 3000, 40, path)
roll("binary", "turtle", (7, 5), 1500, 40, "inc")
roll("binary", "wide", (16, 16), 2000, 30, "incfused", obs_window=(16, 16), controls=["regions", "path-length"])
roll("binary", "narrow", (16, 16), 70000, 6, compact=True)          # chunked host pipeline over the split path
roll("zelda", "turtle", (7, 11), 3000, 40, "split")
roll("binary_holey", "narrow", (16, 16), 2000, 30, "split")
roll("minecraft_2D_maze", "narrow", (14, 14), 2000, 30)
roll("binary", "narrow", (64, 64), 300, 12)
roll("zelda", "turtle", (40, 50), 300, 12)
roll("sokoban", "cellular", (5, 5), 60000, 4, action_kind="ca_tiles")
roll("sokoban", "narrow", (5, 5), 4000, 30)
roll("smb", "narrow", (20, 16), 400, 10)            # lane groups, heap in shared memory
roll("smb", "narrow", (12, 40), 300, 8)             # lane groups, heap continued in the global slice
os.environ["PCGRL_SMB_GROUP_CAP"] = "32"
roll("smb", "narrow", (20, 16), 300, 6)             # most levels overflow the group's slice: whole-warp fallback
os.environ.pop("PCGRL_SMB_GROUP_CAP")
roll("smb", "turtle", (140, 12), 64, 6)             # bit map too tall for a group: every level through the fallback
roll("minecraft_3D_maze", "narrow", (8, 8, 8), 600, 12)
roll("minecraft_3D_holey_maze", "narrow", (7, 7, 7), 500, 12)
roll("minecraft_3D_dungeon_holey", "turtle", (7, 7, 7), 500, 12, fixed_holes=True)


def multiagent():
    cfg = P.make_config("zelda", "turtle", map_shape=(7, 11), obs_window=(22, 22), max_board_scans=0.3)
    cfg.multiagent.n_agents = 3
    env = P.BatchedPcgrlEnv(cfg, 2000, seed=2, auto_reset=True)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(0)
    for t in range(12):
        env.step_agents(torch.randint(0, 4 + env.n_tiles, (2000, 3), generator=g, device=env.device, dtype=torch.int32))
    for a in range(3):
        env.observe(dtype=torch.uint8, agent=a)
    torch.cuda.synchronize()
    env.check_status()
    print("ok multi-agent zelda turtle", flush=True)


multiagent()
print("memcheck workload done")
