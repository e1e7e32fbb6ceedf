#!/usr/bin/env python
"""Time saving, loading and forking packed env rows (pcgrl_save_envs / pcgrl_load_envs, BatchedPcgrlEnv.save_envs /
load_envs / fork_envs) against the torch-index workaround they replace.

    python scripts/bench_env_rows.py [--out profiles/r03_env_rows.jsonl] [--quick]

Workloads (every shard first reset and stepped 24 random steps, so maps, positions and counters are mid-episode):
  a. binary-narrow 16x16, 1 Mi envs     rows with the incremental search's cache row
  b. zelda-turtle 7x11, 64 Ki envs
  c. minecraft_3D_maze 14^3, 64 Ki envs the largest grid row (2 752 bytes)
and M = 1 Ki, 64 Ki and N rows: src a random draw with repeats, dst random distinct, unsorted.  Per (workload, M):
  save_ms / load_ms / fork_ms           the C calls on device indices (fork = save into a buffer, then load);
  py_save_ms / py_load_ms / py_fork_ms  the BatchedPcgrlEnv calls with device indices (they add the index checks'
                                        reductions and syncs, and load_envs its header check);
  workaround_ms                         t[dst] = t[src] over every per-env tensor (what a user writes without fork_envs);
  save_kernel_us / load_kernel_us       kernel times from a torch.profiler pass of their own;
  save_TBps / load_TBps                 2 * S * M bytes (each row byte read once and written once) over kernel time.
Each call is timed alone with CUDA events, with L2 (126 MB) overwritten before it, over --reps calls after a warm one.
Before timing, fork_envs and the workaround start from the same state and must leave the same state
("equal_to_workaround").  Every line carries the GPU name and power limit read in the same run.
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


def _flush():
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    _FLUSH.zero_()


def timed_ms(fn, reps):
    """Mean device time of fn over reps calls, each with L2 overwritten before it and timed alone."""
    fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for e0, e1 in evs:
        _flush()
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    return sum(e0.elapsed_time(e1) for e0, e1 in evs) / reps


def kernel_us(fn, reps, name):
    """Mean device time of the kernel whose name contains `name`, from a torch.profiler run of its own."""
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            _flush()
            fn()
        torch.cuda.synchronize()
    hits = [e for e in prof.key_averages() if name in e.key]
    n = sum(e.count for e in hits)
    return sum(e.device_time_total for e in hits) / n if n else float("nan")


def actions(env, m, g):
    shape, _, tdt = env._action_layout(m)
    return torch.randint(0, env.n_discrete_actions(), shape, generator=g, device=env.device).to(tdt)


def make(problem, rep, shape, n, seed=1):
    env = P.BatchedPcgrlEnv(P.make_config(problem, rep, map_shape=shape), n, seed=seed)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(seed)
    for _ in range(24):
        env.step(actions(env, n, g))
    return env, g


def workaround(env, src, dst):
    """Today's way to copy env rows between slots: index every per-env tensor."""
    for k in STATE:
        t = getattr(env, k)
        if t is None or (k == "targets" and t.shape[0] != env.n_envs):
            continue
        if k == "agent_pos":
            t[:, dst] = t[:, src]
        else:
            t[dst] = t[src]


def same_state(a, b):
    return all(getattr(a, k) is None or torch.equal(getattr(a, k).reshape(-1).view(torch.uint8),
                                                    getattr(b, k).reshape(-1).view(torch.uint8)) for k in STATE)


def bench(a, info, label, problem, rep, shape, n):
    env, g = make(problem, rep, shape, n)
    lib, S, n_pos = env.lib, env.env_row_bytes, env.agent_pos.shape[0]
    for m in sorted({1 << 10, min(64 << 10, n), n}):
        src = torch.randint(0, n, (m,), generator=g, device=env.device).to(torch.int32)
        dst = torch.randperm(n, generator=g, device=env.device)[:m].to(torch.int32)
        src_l, dst_l = src.long(), dst.long()
        # fork_envs and the workaround from the same state
        twin = P.BatchedPcgrlEnv(env.cfg, n, seed=env.seed)
        twin.load_state_dict(env.state_dict())
        for k in ("reward", "done", "changed"):
            getattr(twin, k).copy_(getattr(env, k))
        env.fork_envs(src, dst)
        workaround(twin, src_l, dst_l)
        equal = same_state(env, twin)
        del twin
        torch.cuda.empty_cache()
        rows = torch.empty((m, S), dtype=torch.uint8, device=env.device)
        save = lambda: P._lib.check(lib.pcgrl_save_envs(env._cc, env._st, n_pos, src.data_ptr(), m, rows.data_ptr(),  # noqa: E731
                                                        env._stream()), "save")
        load = lambda: P._lib.check(lib.pcgrl_load_envs(env._cc, env._st, n_pos, rows.data_ptr(), dst.data_ptr(), m,  # noqa: E731
                                                        env._stream()), "load")
        save()
        t_save, t_load = timed_ms(save, a.reps), timed_ms(load, a.reps)
        t_fork = timed_ms(lambda: (save(), load()), a.reps)
        k_save, k_load = kernel_us(save, a.reps, "k_save_envs"), kernel_us(load, a.reps, "k_load_envs")
        t_py_save = timed_ms(lambda: env.save_envs(src), a.reps)
        t_py_load = timed_ms(lambda: env.load_envs(rows, dst), a.reps)
        t_py_fork = timed_ms(lambda: env.fork_envs(src, dst), a.reps)
        t_wa = timed_ms(lambda: workaround(env, src_l, dst_l), a.reps)
        moved = 2 * S * m
        emit({**info, "workload": label, "envs": n, "M": m, "row_bytes": S, "save_ms": round(t_save, 4),
              "load_ms": round(t_load, 4), "fork_ms": round(t_fork, 4), "py_save_ms": round(t_py_save, 4),
              "py_load_ms": round(t_py_load, 4), "py_fork_ms": round(t_py_fork, 4), "workaround_ms": round(t_wa, 4),
              "save_kernel_us": round(k_save, 2), "load_kernel_us": round(k_load, 2),
              "save_TBps": round(moved / (k_save * 1e-6) / 1e12, 3), "load_TBps": round(moved / (k_load * 1e-6) / 1e12, 3),
              "workaround_over_fork": round(t_wa / t_fork, 2), "workaround_over_py_fork": round(t_wa / t_py_fork, 2),
              "equal_to_workaround": bool(equal)}, a.out)
    env.check_status()
    del env
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_env_rows.jsonl"))
    ap.add_argument("--quick", action="store_true", help="1/64 of the shard sizes (a rehearsal, not a measurement)")
    ap.add_argument("--reps", type=int, default=40)
    a = ap.parse_args()
    info = gpu_info()
    div = 64 if a.quick else 1
    bench(a, info, "a: binary-narrow 16x16", "binary", "narrow", (16, 16), (1 << 20) // div)
    bench(a, info, "b: zelda-turtle 7x11", "zelda", "turtle", (7, 11), (64 << 10) // div)
    bench(a, info, "c: minecraft_3D_maze 14^3", "minecraft_3D_maze", "narrow", (14, 14, 14), (64 << 10) // div)


if __name__ == "__main__":
    main()
