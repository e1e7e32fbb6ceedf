#!/usr/bin/env python
"""Device-time the float16 / bfloat16 observation writer against the two ways a half-precision policy got its input
before: observe in float32 and cast, or observe in uint8 and cast (only where there are no target planes).

    python scripts/bench_observe_half.py [--envs N] [--reps R] [--out profiles/r03_observe_half.jsonl]

Shapes (262 144 envs by default, so every output is larger than the 126 MB L2 and no flush is needed):
  binary-narrow 16x16 behind its 32x32 crop; binary-wide 16x16 whole map + controls [regions, path-length];
  zelda-turtle 7x11 behind its 22x22 crop; minecraft_3D_maze narrow 14^3 behind its 14^3 crop.
Each shard is reset, stepped 8 random steps and gets random crop centres.  Every writer and workaround runs into a
preallocated tensor; a workaround's cast also writes into one.  Times come from CUDA events over R calls after warm-up.
"bytes" is what the writer must move (output + grid rows + positions); for a workaround it is the writer's bytes plus
the cast's read and write.  GB/s over MEASURED_PEAKS.json's HBM rate (else the 6 544 GB/s of DESIGN 4.6) is
"frac_of_hbm_peak".  Each half result is also compared, byte for byte, with the float32 observation converted.  Every
line carries the GPU name and power limit read in the same run.
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

SHAPES = [  # (label, problem, rep, map_shape, obs_window, controls)
    ("binary-narrow 16x16, 32x32 crop", "binary", "narrow", (16, 16), (32, 32), None),
    ("binary-wide 16x16 + regions, path-length", "binary", "wide", (16, 16), (16, 16), ["regions", "path-length"]),
    ("zelda-turtle 7x11, 22x22 crop", "zelda", "turtle", (7, 11), (22, 22), None),
    ("minecraft_3D_maze narrow 14^3", "minecraft_3D_maze", "narrow", (14, 14, 14), (14, 14, 14), None),
]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power}


def events_ms(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def make_env(problem, rep, shape, window, controls, n):
    cfg = P.make_config(problem, rep, map_shape=shape, obs_window=window, controls=controls)
    env = P.BatchedPcgrlEnv(cfg, n, seed=1, action_kind="wide_flat" if rep == "wide" else None)
    g = torch.Generator(device=env.device).manual_seed(1)
    if controls:
        env.sample_uniform_targets(generator=g)
    env.reset()
    for _ in range(8):
        env.step(torch.randint(0, env.n_discrete_actions(), (n,), generator=g, device=env.device,
                               dtype=env._action_layout()[2]))
    if rep in ("narrow", "turtle"):   # spread the crop centres
        for i, d in enumerate(shape):
            env.pos[:, i] = torch.randint(0, d, (n,), generator=g, device=env.device, dtype=torch.int32)
    return env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 18)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="", help="also append the JSON lines to this file")
    a = ap.parse_args()
    info = gpu_info()
    # without MEASURED_PEAKS.json: the 6 544 GB/s measured on a B200 that DESIGN 4.6 and scripts/bench_observe.py use
    peak, peak_src = 6544.0, "6544 GB/s measured earlier (DESIGN 4.6)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak, peak_src = float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:  # noqa: BLE001
        pass
    info["hbm_peak_source"] = peak_src
    n = a.envs
    for label, problem, rep, shape, window, controls in SHAPES:
        env = make_env(problem, rep, shape, window, controls, n)
        shp = (n, *env.obs_shape())
        read = n * (env.row_stride + 12)
        buf = {dt: torch.empty(shp, dtype=dt, device=env.device)
               for dt in (torch.float16, torch.bfloat16, torch.float32) + (() if controls else (torch.uint8,))}
        cast = torch.empty(shp, dtype=torch.bfloat16, device=env.device)
        runs = [(str(dt).split(".")[-1], lambda dt=dt: env.observe(out=buf[dt]), buf[dt].numel() * buf[dt].element_size() + read)
                for dt in buf]
        for src in (torch.float32,) + (() if controls else (torch.uint8,)):
            nb = buf[src].numel() * buf[src].element_size()
            runs.append((f"{str(src).split('.')[-1]} then .to(bfloat16)",
                         lambda src=src: cast.copy_(env.observe(out=buf[src])), nb + read + nb + cast.numel() * 2))
        times = {}
        for name, fn, nbytes in runs:
            ms = events_ms(fn, a.reps)
            times[name] = ms
            gbs = nbytes / ms / 1e6
            line = {**info, "shape": label, "envs": n, "obs_shape": list(shp[1:]), "writer": name, "ms": round(ms, 4),
                    "bytes": nbytes, "GB/s": round(gbs, 1)}
            line["frac_of_hbm_peak"] = round(gbs / peak, 3)
            if name in ("float16", "bfloat16"):
                dt = getattr(torch, name)
                env.observe(out=buf[torch.float32])
                env.observe(out=buf[dt])
                line["equals_float32_converted"] = bool(torch.equal(buf[dt].view(torch.int16),
                                                                    buf[torch.float32].to(dt).view(torch.int16)))
            print(json.dumps(line), flush=True)
            if a.out:
                with open(a.out, "a") as f:
                    f.write(json.dumps(line) + "\n")
        ws = [k for k in times if "then" in k]
        summary = {**info, "shape": label, "envs": n,
                   **{f"{h}_speedup_vs_{w.split()[0]}_cast": round(times[w] / times[h], 2) for h in ("float16", "bfloat16")
                      for w in ws}}
        print(json.dumps(summary), flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(json.dumps(summary) + "\n")
        del env, buf, cast
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
