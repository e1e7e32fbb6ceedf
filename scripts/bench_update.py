#!/usr/bin/env python
"""Device-time BatchedPcgrlEnv.update (pcgrl_update) against step() on twin envs fed the same actions.

    python scripts/bench_update.py [--reps R] [--episode T] [--out FILE]
Prints one JSON line per case and one per generator episode, plus a first line with the GPU's name and power limit
(read-only nvidia-smi query in the same run).

Timing: CUDA events around R >= 50 calls after warm-up calls of the same shapes.  Two action batches alternate, so
that every cellular call really rewrites the maps (with one batch, every call after the first would find the maps
already equal to the argmax and write nothing).

Working sets: the cellular rows stream the logits and the maps once per call -- 2.1 GB (binary 16x16), 0.5 GB
(sokoban 5x5) and 3.4 GB (smb 116x16) of logits alone, far beyond the 126 MB L2.  The narrow rows touch one grid
sector, pos, n_step, the action and `changed` per env: about 55 MB (binary 16x16, 1 Mi envs) and 4 MB (minecraft
14^3, 64 Ki envs) of sectors, which can stay in L2 from call to call, as they do in a generator loop.

Byte model of the cellular rows, from the shapes: logits read (4 C cells) + grid read and written (2 cells) +
changed (1) per env; GB/s and the fraction of the 6.54 TB/s HBM figure scripts/bench_observe.py uses.
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

HBM_GBS = 6544.0
CASES = [  # (problem, rep, map_shape, envs)
    ("binary", "cellular", (16, 16), 1 << 20),
    ("sokoban", "cellular", (5, 5), 1 << 20),
    ("smb", "cellular", (116, 16), 1 << 16),
    ("minecraft_3D_maze", "narrow", (14, 14, 14), 1 << 16),
    ("binary", "narrow", (16, 16), 1 << 20),
]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = [s.strip() for s in out[0].split(",")]
    except Exception as exc:  # noqa: BLE001 -- report what is missing instead of inventing it
        name, power = torch.cuda.get_device_name(0), f"unknown ({exc.__class__.__name__})"
    return {"gpu": name, "power_limit": power}


def random_actions(env, gen):
    n, C = env.n_envs, env.n_tiles
    if env.action_kind == "ca_logits":
        return torch.randn((n, C * env.cells), generator=gen, device=env.device)
    hi = {"narrow": C, "turtle": 4 + C}[env.representation]
    return torch.randint(0, hi, (n,), generator=gen, device=env.device, dtype=torch.int32)


def timed(fn, acts, reps):
    for i in range(4):
        fn(acts[i % 2])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(acts[i % 2])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--episode", type=int, default=50, help="T: update() calls per generator episode")
    ap.add_argument("--cases", default="", help="comma-separated case indices (default: all)")
    ap.add_argument("--out", default="", help="also append the JSON lines to this file")
    a = ap.parse_args()
    if a.reps < 50:
        raise SystemExit("--reps must be >= 50")
    if not torch.cuda.is_available():
        raise SystemExit("bench_update.py times the GPU kernels: no CUDA device")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")

    info = gpu_info()
    emit(info)
    pick = [int(i) for i in a.cases.split(",")] if a.cases else range(len(CASES))
    for ci in pick:
        problem, rep, shape, n = CASES[ci]
        cfg = P.make_config(problem, rep, map_shape=shape)   # no auto-reset: step keeps editing past done
        su, st = P.BatchedPcgrlEnv(cfg, n, seed=1), P.BatchedPcgrlEnv(cfg, n, seed=1)
        su.reset()
        st.reset()
        gen = torch.Generator(device=su.device).manual_seed(0)
        acts = [random_actions(su, gen) for _ in range(2)]
        ms_u = timed(su.update, acts, a.reps)
        ms_s = timed(st.step, acts, a.reps)
        torch.cuda.synchronize()
        case = f"{problem}-{rep}-{'x'.join(map(str, shape))}"
        d = {"case": case, "action_kind": su.action_kind, "envs": n, "reps": a.reps, "update_ms": round(ms_u, 4),
             "step_ms": round(ms_s, 4), "step_over_update": round(ms_s / ms_u, 1),
             "maps_equal_after_same_calls": bool(torch.equal(su.grids, st.grids)), **info}
        if rep == "cellular":
            per_env = 4 * su.n_tiles * su.cells + 2 * su.cells + 1
            gbs = per_env * n / ms_u / 1e6
            d.update({"bytes_per_env": per_env, "update_GB/s": round(gbs, 1), "frac_of_hbm": round(gbs / HBM_GBS, 3),
                      "hbm_figure_GB/s": HBM_GBS})
        emit(d)

        # generator episode: T update() calls + one compute_stats, against T step() calls
        su.reset()
        st.reset()
        T = a.episode

        def ep_update():
            for i in range(T):
                su.update(acts[i % 2])
            return su.compute_stats(su.maps, holes=su.holes)

        def ep_step():
            for i in range(T):
                st.step(acts[i % 2])

        for fn in (ep_update, ep_step):
            fn()
        su.reset()
        st.reset()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        stats_u = ep_update()
        ev[1].record()
        ev[2].record()
        ep_step()
        ev[3].record()
        torch.cuda.synchronize()
        ms_eu, ms_es = ev[0].elapsed_time(ev[1]), ev[2].elapsed_time(ev[3])
        emit({"case": case, "episode": f"{T} x update + compute_stats vs {T} x step", "envs": n,
              "update_episode_ms": round(ms_eu, 3), "step_episode_ms": round(ms_es, 3),
              "speedup": round(ms_es / ms_eu, 1), "final_stats_equal": bool(torch.equal(stats_u, st.stats)), **info})
        del su, st, acts
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
