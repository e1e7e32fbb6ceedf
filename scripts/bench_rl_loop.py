#!/usr/bin/env python
"""Device-time the RL-side loop: PcgrlVectorEnv.step (fused env step + auto-reset) + the observation of every env,
every step, all on the GPU (what a policy that lives on the same device consumes).
    python scripts/bench_rl_loop.py [--envs N] [--steps K] [--obs uint8 float32 bfloat16 codes] [--shards 1 2 4]
                                    [--config binary-narrow | binary-wide-ctrl]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import control_pcgrl_b200 as P  # noqa: E402
from control_pcgrl_b200.vector_env import PcgrlVectorEnv  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=1 << 20)
# default: two whole 770-step episodes, so the number includes the auto-resets (and would expose a per-step
# device-to-host sync after the first episode boundary)
ap.add_argument("--steps", type=int, default=1600)
ap.add_argument("--shards", type=int, nargs="+", default=[1, 2],
                help="env ranges stepped + observed on their own streams (PcgrlVectorEnv(shards=k)); one line per value")
ap.add_argument("--obs", nargs="+", default=["uint8", "float32", "codes"],
                help="uint8 / float32 / float16 / bfloat16: one-hot crops; codes: the crop's tile codes, 1 byte per pixel "
                     "(PcgrlVectorEnv(onehot=False))")
# binary-wide-ctrl: BASELINE config 2, the whole 16x16 map with [regions, path-length] target planes (no uint8)
ap.add_argument("--config", default="binary-narrow", choices=["binary-narrow", "binary-wide-ctrl"])
a = ap.parse_args()
for obs, shards in [(o, k) for o in a.obs for k in a.shards]:
    wide = a.config == "binary-wide-ctrl"
    cfg = P.make_config("binary", "wide", controls=["regions", "path-length"]) if wide else P.make_config("binary", "narrow")
    env = PcgrlVectorEnv(cfg, a.envs, shards=shards, onehot=obs != "codes",
                         obs_dtype=torch.uint8 if obs == "codes" else getattr(torch, obs))
    env.reset()
    acts = torch.randint(0, env.single_action_space.n, (a.steps + 5, a.envs), device=env.env.device, dtype=torch.int32)
    for t in range(5):
        env.step(acts[t])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(a.steps):
        env.step(acts[5 + t])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    if not wide:
        assert env.env._synced_steps is not None, "lost the sync-free episode-end detection"
    print(json.dumps({"loop": f"PcgrlVectorEnv.step + observe, {a.config} 16x16", "obs": obs, "envs": a.envs,
                      "shards": shards, "steps": a.steps, "episode_steps": int(env.env.max_iterations) + 1,
                      "ms_per_step": round(ms, 4), "env_steps_per_s": round(a.envs / ms * 1e3)}), flush=True)
    del env
    torch.cuda.empty_cache()
