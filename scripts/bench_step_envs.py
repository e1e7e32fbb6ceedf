#!/usr/bin/env python
"""Time stepping a subset of envs (pcgrl_step_envs, BatchedPcgrlEnv.step(env_ids=...)) against the full step of the same
shard and against the workaround it replaces.

    python scripts/bench_step_envs.py [--out profiles/r03_step_envs.jsonl] [--quick]

Workloads (every shard first reset and stepped 24 random steps, so maps, positions and counters are mid-episode):
  a. binary-narrow 16x16, 1 Mi envs     indexed path, incremental search
  b. binary-wide 16x16, 64 Ki envs      indexed path, incremental search
  c. zelda-turtle 7x11, 64 Ki envs      indexed path, static search
  d. binary-cellular 16x16, 1 Mi envs   generic path (gather, step, scatter)
  e. minecraft_3D_maze 14^3, 64 Ki envs generic path
and M = 1 Ki, N/16, N/2 and N listed envs (random, distinct, unsorted).  Per (workload, M):
  step_envs_ms    the C call (pcgrl_step_envs) on device indices;
  python_ms       BatchedPcgrlEnv.step(actions, env_ids=ids) with device ids (adds the index check: one sort, one sync);
  full_step_ms    pcgrl_step of all N envs;
  workaround_ms   state_dict() clone, full step, unlisted rows of every state tensor copied back.
Each call is timed alone with CUDA events, with L2 (126 MB) overwritten before it, over --reps calls after a warm one.
Before timing, the subset step and the workaround start from the same state and must leave the same state and
outputs ("equal_to_workaround").  Every line carries the GPU name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import control_pcgrl_b200 as P  # noqa: E402

STATE = ("grids", "agent_pos", "n_step", "iteration", "changes", "stats", "targets", "static_mask", "holes", "records",
         "cache", "reward", "done", "changed")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power}


def emit(line, out):
    s = json.dumps(line)
    print(s, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(s + "\n")


_FLUSH = None


def timed_ms(fn, reps):
    """Mean device time of fn over reps calls, each with L2 overwritten before it and timed alone."""
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for e0, e1 in evs:
        _FLUSH.zero_()
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    return sum(e0.elapsed_time(e1) for e0, e1 in evs) / reps


def actions(env, m, g):
    shape, _, tdt = env._action_layout(m)
    if env.action_kind == "ca_logits":
        return torch.randn(shape, generator=g, device=env.device).contiguous()
    return torch.randint(0, env.n_discrete_actions(), shape, generator=g, device=env.device).to(tdt)


def make(problem, rep, shape, n, seed=1):
    window = {"obs_window": shape} if rep == "wide" else {}
    env = P.BatchedPcgrlEnv(P.make_config(problem, rep, map_shape=shape, **window), n, seed=seed)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(seed)
    for _ in range(24):
        env.step(actions(env, n, g))
    return env, g


def workaround(env, ids, keep, acts_full):
    """Today's way to advance only the listed envs: clone the state, step all, copy the unlisted rows back."""
    sd = env.state_dict()
    old = {k: getattr(env, k).clone() for k in ("reward", "done", "changed")}
    env.step(acts_full)
    for k in STATE:
        t = getattr(env, k)
        if t is None or (k == "targets" and t.shape[0] != env.n_envs):
            continue
        src = old[k] if k in old else sd[k]
        if k == "agent_pos":
            t[:, keep] = src[:, keep]
        else:
            t[keep] = src[keep]


def same_state(a, b):
    return all(getattr(a, k) is None or torch.equal(getattr(a, k).reshape(-1).view(torch.uint8),
                                                    getattr(b, k).reshape(-1).view(torch.uint8)) for k in STATE)


def bench(a, info, label, problem, rep, shape, n):
    env, g = make(problem, rep, shape, n)
    lib = env.lib
    path = "indexed" if env.worklist is not None else "generic"
    full = actions(env, n, g)
    t_full = timed_ms(lambda: P._lib.check(lib.pcgrl_step(env._cc, env._st, full.data_ptr(), env._stream())), a.reps)
    rng = np.random.default_rng(7)
    for m in sorted({1 << 10, n // 16, n // 2, n}):
        ids = torch.from_numpy(rng.permutation(n)[:m].astype(np.int32)).to(env.device)
        keep = torch.ones(n, dtype=torch.bool, device=env.device)
        keep[ids.long()] = False
        acts = actions(env, m, g)
        acts_full = full.clone()
        acts_full[ids.long()] = acts
        # the subset step and the workaround from the same state
        twin = P.BatchedPcgrlEnv(env.cfg, n, seed=env.seed, split_step=env.worklist is not None)
        twin.load_state_dict(env.state_dict())
        for k in ("reward", "done", "changed"):
            getattr(twin, k).copy_(getattr(env, k))
        r, d = env.step(acts, env_ids=ids)
        workaround(twin, ids, keep, acts_full)
        equal = same_state(env, twin) and torch.equal(r.view(torch.int32), twin.reward[ids.long()].view(torch.int32))
        equal = equal and torch.equal(d, twin.done[ids.long()])
        del twin
        torch.cuda.empty_cache()
        work = env._work(int(lib.pcgrl_step_envs_work_bytes(env._cc, m)))
        t_sub = timed_ms(lambda: P._lib.check(lib.pcgrl_step_envs(env._cc, env._st, acts.data_ptr(), ids.data_ptr(), m,
                                                                  work.data_ptr(), env._stream())), a.reps)
        t_py = timed_ms(lambda: env.step(acts, env_ids=ids), a.reps)
        t_wa = timed_ms(lambda: workaround(env, ids, keep, acts_full), max(3, a.reps // 4))
        emit({**info, "workload": label, "path": path, "envs": n, "M": m, "step_envs_ms": round(t_sub, 4),
              "python_ms": round(t_py, 4), "full_step_ms": round(t_full, 4), "workaround_ms": round(t_wa, 4),
              "vs_full_step": round(t_sub / t_full, 3), "speedup_vs_workaround": round(t_wa / t_sub, 1),
              "M_env_steps/s": float(f"{m / t_sub * 1e3 / 1e6:.4g}"), "equal_to_workaround": bool(equal)}, a.out)
    del env
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_step_envs.jsonl"))
    ap.add_argument("--quick", action="store_true", help="1/64 of the shard sizes (a rehearsal, not a measurement)")
    ap.add_argument("--reps", type=int, default=40)
    a = ap.parse_args()
    info = gpu_info()
    div = 64 if a.quick else 1
    bench(a, info, "a: binary-narrow 16x16", "binary", "narrow", (16, 16), (1 << 20) // div)
    bench(a, info, "b: binary-wide 16x16", "binary", "wide", (16, 16), (64 << 10) // div)
    bench(a, info, "c: zelda-turtle 7x11", "zelda", "turtle", (7, 11), (64 << 10) // div)
    bench(a, info, "d: binary-cellular 16x16", "binary", "cellular", (16, 16), (1 << 20) // div)
    bench(a, info, "e: minecraft_3D_maze 14^3", "minecraft_3D_maze", "narrow", (14, 14, 14), (64 << 10) // div)


if __name__ == "__main__":
    main()
