#!/usr/bin/env python
"""Time the lookahead with the observation (pcgrl_lookahead_obs: BatchedPcgrlEnv.lookahead_all / lookahead with
obs_dtype) against the workaround it replaces: copy the candidates' envs into a twin env, step it and observe it.

    python scripts/bench_lookahead_obs.py [--out profiles/r03_lookahead_obs.jsonl] [--quick]

Workloads (every shard first reset and stepped 24 random steps, so maps, positions and counters are mid-episode):
  a. binary-narrow 16x16, lookahead_all of 1 Mi envs x 2 actions (incremental path), uint8 and float32 one-hot;
  b. zelda-turtle 7x11, lookahead_all of 64 Ki envs x 12 actions (generic path), uint8 and float32 one-hot;
  c. minecraft_3D_maze narrow 14x14x14, lookahead of a chosen subset: one random action for each of 16 Ki envs, uint8.
The workaround: save the candidates' env rows into a preallocated buffer, load them into a twin env with one slot per
candidate, step every slot, observe every slot into a preallocated tensor; its outputs are compared with the lookahead's
(they must be equal).  Times come from CUDA events around synchronised work, after one warm call.  A torch.profiler run
of its own gives the kernel times; "obs_TB/s" is the observation bytes written over the observation kernel's time.
Every line carries the GPU name and power limit read in the same run.
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch  # noqa: E402
import control_pcgrl_b200 as P  # noqa: E402
from bench_lookahead import emit, events_ms, gpu_info, kernel_ms, make  # noqa: E402


def twin_workaround(env, ids, acts, dtype):
    """-> (fn, outputs): fn re-runs save rows -> load into the twin -> step -> observe."""
    m = ids.numel()
    twin = P.BatchedPcgrlEnv(env.cfg, m, seed=env.seed, split_step=env.worklist is not None)
    rows = torch.empty((m, env.env_row_bytes), dtype=torch.uint8, device=env.device)
    obs = torch.empty((m, *env.obs_shape()), dtype=dtype, device=env.device)

    def run():
        env._save_rows(ids, m, rows)
        twin._load_rows(rows, None, m)
        twin.step(acts)
        twin.observe(out=obs)

    run()
    return run, (twin.reward, twin.done, twin.stats, twin.changed, obs)


def bench(a, info, label, env, ids, acts, dtype):
    m = ids.numel()
    path = "incremental" if env.cache is not None else "generic"
    A = env.n_discrete_actions()
    if ids.numel() == env.n_envs * A:    # every action of every env: lookahead_all
        def call():
            return env.lookahead_all(obs_dtype=dtype)
    else:
        def call():
            return env.lookahead(acts, env_ids=ids, obs_dtype=dtype)
    res = call()
    ms = events_ms(call, a.reps)
    obs_bytes = res[4].numel() * res[4].element_size()
    line = {**info, "workload": label, "path": path, "dtype": str(dtype).replace("torch.", ""), "candidates": m,
            "obs_bytes_per_candidate": obs_bytes // m, "ms": round(ms, 3),
            "candidates/s": float(f"{m / ms * 1e3:.4g}"), "obs_bytes/call_time_TB/s": round(obs_bytes / ms / 1e9, 3)}
    kt = kernel_ms(call, 3)
    line["kernel_ms"] = kt
    ok = sum(v for k, v in kt.items() if k.startswith("k_observe"))
    if ok:
        line["obs_TB/s"] = round(obs_bytes / ok / 1e9, 3)
    run, want = twin_workaround(env, ids, acts, dtype)
    tms = events_ms(run, 1 if a.quick else 3)
    got = [res[0].reshape(m), res[1].reshape(m), res[2].reshape(m, env.K), res[3].reshape(m), res[4].reshape(want[4].shape)]
    line["twin_ms"] = round(tms, 3)
    line["speedup_vs_twin"] = round(tms / ms, 2)
    line["equal_to_twin"] = bool(torch.equal(got[0].view(torch.int32), want[0].view(torch.int32)) and
                                 all(torch.equal(x, y) for x, y in zip(got[1:], want[1:])))
    emit(line, a.out)
    del res, got, want, run
    torch.cuda.empty_cache()


def all_pairs(env):
    """lookahead_all's candidate order: env-major, action a in column a."""
    A = env.n_discrete_actions()
    c = torch.arange(env.n_envs * A, dtype=torch.int32, device=env.device)
    return (c // A).contiguous(), (c % A).to(env._action_layout()[2]).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lookahead_obs.jsonl"))
    ap.add_argument("--quick", action="store_true", help="1/64 of the shard sizes (a rehearsal, not a measurement)")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    info = gpu_info()
    div = 64 if a.quick else 1
    env = make("binary", "narrow", (16, 16), (1 << 20) // div)
    for dtype in (torch.uint8, torch.float32):
        bench(a, info, "a: binary-narrow 16x16, lookahead_all", env, *all_pairs(env), dtype)
    del env
    torch.cuda.empty_cache()
    env = make("zelda", "turtle", (7, 11), (64 << 10) // div)
    for dtype in (torch.uint8, torch.float32):
        bench(a, info, "b: zelda-turtle 7x11, lookahead_all", env, *all_pairs(env), dtype)
    del env
    torch.cuda.empty_cache()
    env = make("minecraft_3D_maze", "narrow", (14, 14, 14), (16 << 10) // div)
    g = torch.Generator(device=env.device).manual_seed(3)
    ids = torch.arange(env.n_envs, dtype=torch.int32, device=env.device)
    acts = torch.randint(0, env.n_discrete_actions(), (env.n_envs,), generator=g, device=env.device, dtype=torch.int32)
    bench(a, info, "c: minecraft_3D_maze 14x14x14, one action per env", env, ids, acts, torch.uint8)


if __name__ == "__main__":
    main()
