#!/usr/bin/env python
"""Time the one-step lookahead (BatchedPcgrlEnv.lookahead_all, pcgrl_lookahead) against the twin-env loop it replaces.

    python scripts/bench_lookahead.py [--out profiles/r03_lookahead.jsonl] [--quick]

Workloads (every shard first reset and stepped 24 random steps, so maps, positions and counters are mid-episode):
  a. binary-narrow 16x16, lookahead_all of 1 Mi envs (2 Mi candidates; incremental path);
  b. binary-wide 16x16 (ActionMap 16 x 16), all 512 actions of 16 Ki envs (8 Mi candidates, two launches of 4 Mi),
     on the incremental path and on the generic path (the same env built with split_step=False);
  c. zelda-turtle 7x11, all 12 actions of 64 Ki envs (generic path);
  and for b and c the loop it replaces: A x (load_state_dict into a twin env + step), whose outputs are also compared
  with the lookahead's (they must be equal).
Times come from CUDA events around synchronised work, after one warm call.  A torch.profiler run of its own gives the
kernel times; the gather kernel's bytes/s counts the bytes it must move (rows read and written, from the shapes).
Every line carries the GPU name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import control_pcgrl_b200 as P  # noqa: E402


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


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_ms(fn, reps):
    """Device time per call of every kernel fn launches (torch.profiler, CUDA activities)."""
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        if t and "k_" in ev.key:
            name = ev.key.split("(")[0].replace("void ", "").replace("pcgrl::", "")
            out[name] = round(out.get(name, 0) + t / 1e3 / reps, 4)
    return out


def make(problem, rep, shape, n, seed=1, **kw):
    window = {"obs_window": shape} if rep == "wide" else {}
    env = P.BatchedPcgrlEnv(P.make_config(problem, rep, map_shape=shape, **window), n, seed=seed, **kw)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(seed)
    for _ in range(24):
        env.step(torch.randint(0, env.n_discrete_actions(), (n,), generator=g, device=env.device, dtype=torch.int32))
    return env


def gather_bytes(env, m):
    """Bytes k_la_gather must move for m candidates: every row it reads from the shard and writes to the sub-shard."""
    rows = env.row_stride * (2 if env.static_mask is not None else 1) + 12 + 12 + 4 * env.K
    rows += 16 * env.K if env.ctrl_metrics else 0
    rows += 4 * env.hole_ints if env.holey else 0
    return m * (2 * rows + 4)


def twin_table(env, reps):
    """The loop the lookahead replaces: per action a, restore a twin from the env's state and step every env with a."""
    A = env.n_discrete_actions()
    twin = P.BatchedPcgrlEnv(env.cfg, env.n_envs, seed=env.seed, split_step=env.worklist is not None)
    sd = env.state_dict()
    tdt = env._action_layout()[2]
    acts = [torch.full((env.n_envs,), a, device=env.device, dtype=torch.int32).to(tdt) for a in range(A)]
    reward = torch.empty((env.n_envs, A), dtype=torch.float32, device=env.device)
    stats = torch.empty((env.n_envs, A, env.K), dtype=torch.int32, device=env.device)

    def run():
        for a in range(A):
            twin.load_state_dict(sd)
            r, _ = twin.step(acts[a])
            reward[:, a] = r
            stats[:, a] = twin.stats

    ms = events_ms(run, reps)
    return ms, reward, stats


def bench(a, info, label, env, twin=True):
    A = env.n_discrete_actions()
    m = env.n_envs * A
    path = "incremental" if env.cache is not None else "generic"
    res = env.lookahead_all()
    ms = events_ms(env.lookahead_all, a.reps)
    changed = float(res[3].float().mean())
    line = {**info, "workload": label, "path": path, "envs": env.n_envs, "actions": A, "candidates": m,
            "ms": round(ms, 3), "candidates/s": float(f"{m / ms * 1e3:.4g}"), "changed_share": round(changed, 4),
            "changed/s": float(f"{m * changed / ms * 1e3:.4g}")}
    kt = kernel_ms(env.lookahead_all, 3)
    line["kernel_ms"] = kt
    gk = sum(v for k, v in kt.items() if k.startswith("k_la_gather"))
    if gk:
        line["gather_GB/s"] = round(gather_bytes(env, m) / gk / 1e6, 1)
    sk = sum(v for k, v in kt.items() if k.startswith("k_split_stats_inc"))
    if sk:
        line["search_us_per_Mi_changed"] = round(sk * 1e3 / (m * changed / (1 << 20)), 1)
    if twin:
        tms, tr, ts = twin_table(env, 1 if a.quick else 3)
        line["twin_loop_ms"] = round(tms, 3)
        line["speedup_vs_twin"] = round(tms / ms, 2)
        line["equal_to_twin"] = bool(torch.equal(tr.view(torch.int32), res[0].view(torch.int32)) and torch.equal(ts, res[2]))
    emit(line, a.out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lookahead.jsonl"))
    ap.add_argument("--quick", action="store_true", help="1/64 of the shard sizes (a rehearsal, not a measurement)")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    info = gpu_info()
    div = 64 if a.quick else 1
    bench(a, info, "a: binary-narrow 16x16, lookahead_all", make("binary", "narrow", (16, 16), (1 << 20) // div))
    for split in (True, False):
        env = make("binary", "wide", (16, 16), (16 << 10) // div, split_step=split)
        bench(a, info, "b: binary-wide 16x16, 512 actions", env)
        del env
        torch.cuda.empty_cache()
    bench(a, info, "c: zelda-turtle 7x11, 12 actions", make("zelda", "turtle", (7, 11), (64 << 10) // div))


if __name__ == "__main__":
    main()
