#!/usr/bin/env python
"""Time the observation of a list of envs (pcgrl_observe_envs) and the two seams that use it.

    python scripts/bench_observe_envs.py [--out profiles/r03_observe_envs.jsonl] [--quick]

1. writer: observe(env_ids=idx) of M rows at N = 1 Mi binary-narrow (u8 one-hot, f32, tile codes) and 256 Ki
   zelda-turtle u8, M in {1, 64, 4096, 65536, N/2, N}, ascending and shuffled indices, against the full observe() of
   the same shard in the same run (CUDA events; GB/s counts the M rows written).
2. PcgrlVectorEnv.step at 64 Ki and 1 Mi envs with change_percentage=0.2 (episodes end at different steps), with the
   final observations and with the step of the parent commit (no final observations), alternating in one process.
3. vector_step of the RLlib seam at 4 Ki and 64 Ki envs, change_percentage=0.2: the rows-only observe / download
   against the parent's full observe + full download, alternating; device-to-host bytes counted from the copies made.
Every line carries the GPU name and power limit read in the same run.  Outputs of the timed cases are larger than L2
(126 MB) except for small M, which measures launch overhead.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import control_pcgrl_b200 as P  # noqa: E402
from control_pcgrl_b200.vector_env import PcgrlVectorEnv  # noqa: E402


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


def bench_writer(a, info):
    cases = [("binary", "narrow", (16, 16), (32, 32), torch.uint8, True, 1 << 20),
             ("binary", "narrow", (16, 16), (32, 32), torch.float32, True, 1 << 20),
             ("binary", "narrow", (16, 16), (32, 32), torch.uint8, False, 1 << 20),
             ("zelda", "turtle", (7, 11), (22, 22), torch.uint8, True, 1 << 18)]
    for problem, rep, shape, window, dt, onehot, n in cases:
        if a.quick:
            n //= 64
        env = P.BatchedPcgrlEnv(P.make_config(problem, rep, map_shape=shape, obs_window=window), n, seed=1)
        env.reset()
        for i, d in enumerate(shape):
            env.pos[:, i] = torch.randint(0, d, (n,), device=env.device, dtype=torch.int32)
        out = torch.empty((n, *env.obs_shape(onehot)), dtype=dt, device=env.device)
        row_bytes = out[0].numel() * out.element_size()
        ms_full = events_ms(lambda: env.observe(out=out, onehot=onehot), a.reps)
        base = {**info, "bench": "writer", "case": f"{problem}-{rep}-{'x'.join(map(str, shape))}",
                "dtype": str(dt).split(".")[-1] + ("" if onehot else " tile codes"), "envs": n,
                "full_ms": round(ms_full, 4), "full_GB/s": round(n * row_bytes / ms_full / 1e6, 1)}
        gen = torch.Generator(device=env.device).manual_seed(0)
        for m in (1, 64, 4096, 65536, n // 2, n):
            if m > n:
                continue
            for order in ("ascending", "shuffled"):
                if order == "ascending":
                    idx = torch.arange(m, dtype=torch.int32, device=env.device)
                else:
                    idx = torch.randperm(n, generator=gen, device=env.device)[:m].to(torch.int32)
                o = out[:m]
                ms = events_ms(lambda: env._observe_envs(idx, out=o, onehot=onehot), a.reps)
                emit({**base, "M": m, "order": order, "ms": round(ms, 4),
                      "GB/s": round(m * row_bytes / ms / 1e6, 1), "ms_vs_full": round(ms / ms_full, 4)}, a.out)
        del env, out
        torch.cuda.empty_cache()


def _step_shard_parent(self, b, actions, lo, hi, infos):
    """PcgrlVectorEnv._step_shard of the parent commit: auto-reset without final observations."""
    reward, done = b.step(actions)
    ret, length = self.episode_return[lo:hi], self.episode_length[lo:hi]
    ret += reward.double()
    length += 1
    lock_step = b.max_changes is None and b._synced_steps is not None
    any_done = (b._synced_steps > b.max_iterations) if lock_step else bool(done.any())
    if any_done:
        d = done.bool()
        infos.append((lo, {"final_stats": b.stats.clone(), "final_return": ret.clone(),
                           "final_length": length.clone(), "_final": d}))
        if lock_step:
            b.reset()
            ret.zero_()
            length.zero_()
        else:
            b.reset(mask=done)
            ret[d] = 0
            length[d] = 0
    b.observe(out=self._obs[lo:hi], onehot=self.onehot)
    return reward, done


def bench_vector_step(a, info):
    for n in ((1 << 16, 1 << 20) if not a.quick else (1 << 12,)):
        cfg = P.make_config("binary", "narrow", change_percentage=0.2)
        venv = PcgrlVectorEnv(cfg, n, seed=3, obs_dtype=torch.float32)
        venv.reset()
        gen = torch.Generator(device=venv.env.device).manual_seed(0)
        acts = [torch.randint(0, 2, (n,), generator=gen, device=venv.env.device, dtype=torch.int32) for _ in range(8)]
        arms = {"final_obs": PcgrlVectorEnv._step_shard, "parent": _step_shard_parent}
        times = {k: [] for k in arms}
        finals = []
        for _ in range(a.warmup):
            venv.step(acts[0])
        for r in range(a.rounds):
            for name, fn in arms.items():
                venv._step_shard = fn.__get__(venv)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for k in range(a.steps):
                    _, _, _, _, inf = venv.step(acts[k % len(acts)])
                    if name == "final_obs" and inf:
                        finals.append(int(inf["final_idx"].numel()))
                torch.cuda.synchronize()
                times[name].append((time.perf_counter() - t0) / a.steps * 1e3)
        emit({**info, "bench": "PcgrlVectorEnv.step", "case": "binary-narrow-16x16 change_percentage=0.2 f32",
              "envs": n, "steps_per_round": a.steps, "rounds": a.rounds,
              "ms_per_step_final_obs": [round(x, 3) for x in times["final_obs"]],
              "ms_per_step_parent": [round(x, 3) for x in times["parent"]],
              "median_final_obs": round(float(np.median(times["final_obs"])), 3),
              "median_parent": round(float(np.median(times["parent"])), 3),
              "mean_finished_per_step": round(float(np.mean(finals)) if finals else 0.0, 1)}, a.out)
        del venv, acts
        torch.cuda.empty_cache()


def bench_rllib(a, info):
    for n in ((1 << 12, 1 << 16) if not a.quick else (1 << 10,)):
        cfg = P.make_config("binary", "narrow", change_percentage=0.2, controls=["regions"])
        venv = P.make_rllib_vector_env(cfg, n, seed=4, obs_dtype=np.float32)
        venv.vector_reset()
        row_bytes = int(np.prod(venv.observation_space.shape)) * 4
        d2h = {"rows": 0, "parent": 0}
        arm = ["rows"]
        new_rows_into = venv._observe_rows_into

        def parent_rows_into(ids, host):      # the parent commit: a full observe and a full download
            venv._observe_into(host)
            venv._new_row[:] = np.arange(venv.num_envs)

        def counted_rows_into(ids, host):
            d2h[arm[0]] += (len(ids) if arm[0] == "rows" else venv.num_envs) * row_bytes
            (new_rows_into if arm[0] == "rows" else parent_rows_into)(ids, host)

        venv._observe_rows_into = counted_rows_into
        rng = np.random.default_rng(0)
        acts = [rng.integers(0, 2, size=n).tolist() for _ in range(8)]
        times = {"rows": [], "parent": []}
        steps = {"rows": 0, "parent": 0}
        for _ in range(a.warmup):
            venv.vector_step(acts[0])
        for r in range(a.rounds):
            for name in ("rows", "parent"):
                arm[0] = name
                t0 = time.perf_counter()
                for k in range(a.steps):
                    venv.vector_step(acts[k % len(acts)])
                times[name].append((time.perf_counter() - t0) / a.steps * 1e3)
                steps[name] += a.steps
                venv._fresh[:] = False
        d2h_terminal = n * row_bytes      # the terminal observations of every step, both arms
        emit({**info, "bench": "rllib.vector_step", "case": "binary-narrow-16x16 controls=regions change_percentage=0.2 f32",
              "envs": n, "steps_per_round": a.steps, "rounds": a.rounds,
              "ms_per_step_rows": [round(x, 3) for x in times["rows"]],
              "ms_per_step_parent": [round(x, 3) for x in times["parent"]],
              "median_rows": round(float(np.median(times["rows"])), 3),
              "median_parent": round(float(np.median(times["parent"])), 3),
              "obs_d2h_bytes_per_step_rows": round(d2h_terminal + d2h["rows"] / steps["rows"]),
              "obs_d2h_bytes_per_step_parent": round(d2h_terminal + d2h["parent"] / steps["parent"])}, a.out)
        del venv
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_observe_envs.jsonl"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--quick", action="store_true", help="small sizes (a dry run of the script)")
    ap.add_argument("--only", default="writer,step,rllib")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_observe_envs.py measures on a CUDA device; none found")
    info = gpu_info()
    only = set(a.only.split(","))
    if "writer" in only:
        bench_writer(a, info)
    if "step" in only:
        bench_vector_step(a, info)
    if "rllib" in only:
        bench_rllib(a, info)


if __name__ == "__main__":
    main()
