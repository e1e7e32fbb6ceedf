#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched PCGRL step on B200 (the BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--envs E]
                    [--no-configs] [--dump-outputs DIR]

One "step" = one pass of the hot path (pcgrl_step: representation update -> get_stats -> reward) over the
rank's whole env shard, with random actions, plus the auto-reset launches that episodes ending inside the
timed region cause.  Prints ONE JSON line on rank 0 (see the task contract):
  value     whole-job env-steps/s, actions already resident in HBM (device-timed, max over ranks)
  e2e       same metric through the public host-buffer API (BatchedPcgrlEnv.step_host -> pcgrl_step_host):
            actions H2D from pinned memory, reward/done/stats D2H, every step, inside the timed region
  roofline  the step's kernels (binary: k_split_act + k_split_stats_inc + k_split_out, the search 80 % of it) vs the
            measured HBM peak: algorithmic bytes per pcgrl_step / event time around it
  cpu_baseline  the oracle (python port of the reference path) timed on this box's host cores (bounded sample)
  configs   the other BASELINE.json configs (binary-wide + controls and zelda-turtle at 65 536 envs, sokoban-cellular,
            smb-narrow, minecraft 14^3), each a short run of the same three measurements (value / e2e / roofline /
            cpu_baseline) on the same N GPUs; skipped with --no-configs or when --workload names one of them
`--impl reference` times the reference's CPU implementation of the same path on all host cores: the real
reference under oracle/refshim.py when a reference tree exists (/root/reference in the build container, the
unmodified pip install under baseline/_ref on the GPU box -- oracle/install_reference.sh), else the oracle port.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (problem, rep, map_shape, obs_window, controls, default envs/GPU)
    "binary-narrow-16x16": ("binary", "narrow", (16, 16), (32, 32), None, 1 << 20),
    "binary-wide-ctrl-16x16": ("binary", "wide", (16, 16), (16, 16), ["regions", "path-length"], 1 << 20),
    "binary-turtle-16x16": ("binary", "turtle", (16, 16), (32, 32), None, 1 << 20),
    "zelda-turtle-7x11": ("zelda", "turtle", (7, 11), (22, 22), None, 1 << 20),
    "zelda-narrow-7x11": ("zelda", "narrow", (7, 11), (22, 22), None, 1 << 20),
    # BASELINE.json configs 4 and 5 (search-based stats: warp-per-grid kernels)
    "minecraft_3D_maze-narrow-14x14x14": ("minecraft_3D_maze", "narrow", (14, 14, 14), (14, 14, 14), None, 1 << 16),
    "sokoban-cellular-5x5": ("sokoban", "cellular", (5, 5), (5, 5), None, 1 << 20),
    "sokoban-narrow-5x5": ("sokoban", "narrow", (5, 5), (10, 10), None, 1 << 20),
    "smb-narrow-116x16": ("smb", "narrow", (116, 16), (32, 32), None, 1 << 18),
}
# BASELINE.json configs 2-5 as (workload, envs per GPU, timed steps, warm-up steps, e2e steps): short runs printed
# under "configs" next to the headline (config 1's shape at 1 Mi envs per GPU)
SECONDARY = [
    ("binary-wide-ctrl-16x16", 1 << 16, 300, 10, 60),
    ("zelda-turtle-7x11", 1 << 16, 300, 10, 60),
    ("sokoban-cellular-5x5", 1 << 20, 12, 3, 4),
    ("smb-narrow-116x16", 1 << 18, 12, 3, 4),
    ("minecraft_3D_maze-narrow-14x14x14", 1 << 16, 30, 3, 8),
]
METRIC = "env-steps/sec"
UNIT = "env-steps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=800,
                    help="timed steps of the headline workload (its e2e arm times at most 200 of them; the secondary "
                         "configs keep their own counts)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="binary-narrow-16x16", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: workload's)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget for the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline workload only")
    ap.add_argument("--int32-io", action="store_true", help="e2e through the int32 ABI (three dense result arrays) "
                    "instead of compact host I/O (uint8 actions, one packed record array)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload returned (rank 0's shard) to "
                         "DIR/<name>.npy, for comparing two builds output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's outputs: it needs --impl b200")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:  # noqa: BLE001
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------- CPU arms
def _cpu_worker(args):
    """profile_env.py-style loop (profile_env.py:121-171): reset; step(random action) until done; repeat."""
    workload, seconds, seed, use_ref = args
    problem, rep, shape, obs_window, controls, _ = WORKLOADS[workload]
    rng = np.random.default_rng(seed)
    from control_pcgrl_b200.config import TASK_DEFAULTS
    weights = TASK_DEFAULTS[problem]["weights"]
    from oracle.pcgrl_oracle import INIT_PROBS, TILES
    n_tiles = len(TILES[problem])
    n_act = {"narrow": n_tiles, "turtle": 4 + n_tiles, "wide": obs_window[0] * obs_window[1] * n_tiles,
             "cellular": 0}[rep]
    steps = 0
    if use_ref:
        from oracle import refshim as R
        cfg = R.make_cfg(problem, rep, shape, obs_window=obs_window, weights=weights, controls=controls)
        # the reference's wrapped stacks are broken upstream for 3D problems and for cellular (SURVEY A-9, A-22):
        # those run the raw env under ControlWrapper
        env = R.make_wrapped_env(cfg, raw_only=(len(shape) == 3 or rep == "cellular"))
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            env.reset()
            done = False
            while not done and time.perf_counter() - t0 < seconds:
                a = rng.random((n_tiles, *shape), dtype=np.float32) if rep == "cellular" else int(rng.integers(n_act))
                _, _, done, _, _ = env.step(a)
                steps += 1
        return steps, time.perf_counter() - t0
    from oracle import pcgrl_oracle as O
    env = O.OracleEnv(problem, rep, shape, weights=weights, controls=controls)
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        p = rng.random(n_tiles)
        grid = rng.choice(n_tiles, size=shape, p=p / p.sum())
        env.reset(grid, pos=[int(rng.random() * s) for s in shape])
        done = False
        while not done and time.perf_counter() - t0 < seconds:
            if rep == "cellular":
                a = rng.random((n_tiles, *shape), dtype=np.float32)
            else:
                a = int(rng.integers(n_act))
            if rep == "wide":
                a = O.actionmap_unravel(a, obs_window[0], obs_window[1], n_tiles)
            _, done, _ = env.step(a)
            steps += 1
    return steps, time.perf_counter() - t0


def cpu_arm(workload, seconds, cores, seed=0):
    """-> (env-steps/s aggregate, kind, cores, sample description)"""
    from oracle import refshim
    use_ref = refshim.available()
    kind = "reference" if use_ref else "port"
    if cores <= 1:
        s, dt = _cpu_worker((workload, seconds, seed, use_ref))
        rate = s / dt
    else:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(cores) as pool:
            res = pool.map(_cpu_worker, [(workload, seconds, seed + i, use_ref) for i in range(cores)])
        rate = sum(s / dt for s, dt in res)
    what = ("real reference stack under oracle/refshim.py" if use_ref else "oracle/pcgrl_oracle.py (python port)")
    sample = (f"{what}; profile_env.py-style random-action episodes of {workload}, one env per process, "
              f"{cores} process(es) x {seconds:.0f}s wall")
    return rate, kind, cores, sample


# ------------------------------------------------------------------------------------------- GPU arms
DUMP_ARRAY_BYTES = 12 << 20     # per array; five arrays stay under 64 MB


def dump_outputs(env, out_dir):
    """What a caller of BatchedPcgrlEnv.step holds after the last timed step (reward and done as returned, then the
    stats, positions and maps, auto-reset applied) as float32 .npy files.  An array larger than DUMP_ARRAY_BYTES
    keeps a fixed sample of env rows: the first k of np.random.default_rng(0).permutation(n_envs), in env order."""
    import torch
    arrays = {"reward": env.reward, "done": env.done, "stats": env.stats, "pos": env.pos[:, :env.ndim],
              "maps": env.maps}
    order = np.random.default_rng(0).permutation(env.n_envs)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        row_bytes = 4 * max(1, t[0].numel())
        k = min(env.n_envs, DUMP_ARRAY_BYTES // row_bytes)
        if k < env.n_envs:
            t = t[torch.from_numpy(np.sort(order[:k])).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))


def run_workload(a, workload, n_envs, steps, warmup, e2e_steps, rank, world, local, clock_sampler=None,
                 dump_dir=None):
    """value / e2e / roofline of one workload on this rank's GPU (max over ranks).  -> dict (same on every rank)"""
    import torch
    import torch.distributed as dist
    import control_pcgrl_b200 as P
    from control_pcgrl_b200 import _lib

    problem, rep, shape, obs_window, controls, _ = WORKLOADS[workload]
    dev = torch.device("cuda", local)
    lib = _lib.load()
    cfg = P.make_config(problem, rep, map_shape=shape, obs_window=obs_window, controls=controls)
    env = P.BatchedPcgrlEnv(cfg, n_envs, device=dev, env_offset=rank * n_envs, seed=a.seed, auto_reset=True,
                            action_kind="ca_tiles" if rep == "cellular" else None,
                            compact_host_io=not a.int32_io)
    if controls:
        env.sample_uniform_targets()
    env.reset()
    n_act = {"narrow": env.n_tiles, "turtle": 4 + env.n_tiles,
             "wide": obs_window[0] * obs_window[1] * env.n_tiles, "cellular": 0}[rep]
    gen = torch.Generator(device=dev).manual_seed(a.seed + rank)
    # one distinct uniform-random action batch per step, all resident in HBM before the timed region.
    # (Cycling a small pool would be wrong: the narrow scan revisits a cell every 256 steps and would replay
    # the same action on it, so nothing would change after the first board scan.)
    shape_a, dt_a, tdt_a = env._action_layout()
    bytes_a = int(np.prod(shape_a)) * np.dtype(dt_a).itemsize
    POOL = min(steps + warmup, max(16, int(6e9 // bytes_a)))
    if rep == "cellular":
        # cellular: each action is a whole next map (pre-argmaxed int8 tiles), drawn from the problem's tile
        # distribution so that the solver preconditions of sokoban hold as often as in generated levels
        cdf = torch.tensor(np.cumsum(env.spec.init_probs) / np.sum(env.spec.init_probs), device=dev,
                           dtype=torch.float32)
        act_all = torch.empty((POOL, *shape_a), device=dev, dtype=torch.int8)
        for i in range(POOL):
            u = torch.rand(shape_a, generator=gen, device=dev)
            act_all[i] = torch.searchsorted(cdf, u).clamp_(max=env.n_tiles - 1).to(torch.int8)
            act_all[i, :, env.cells:] = 0
    else:
        act_all = torch.randint(0, n_act, (POOL, n_envs), generator=gen, device=dev, dtype=torch.int32).to(tdt_a)
    act_pool = [act_all[i] for i in range(POOL)]
    step_no = [0]
    # inputs larger than L2 need no flush (the grids alone are 268 MB at the headline size); smaller shards flush
    # 256 MB between steps, outside the timing
    grid_bytes = n_envs * env.row_stride
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if grid_bytes < (200 << 20) else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(k):
        """device-resident arm; returns (sum of per-launch step-kernel ms, total region ms)"""
        evs = []
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(k):
            if flush is not None:
                f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
                f0.record(); flush.fill_(i & 0xFF); f1.record()
                evs.append(("f", f0, f1))
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(lib.pcgrl_step(env._cc, env._st, act_pool[step_no[0] % POOL].data_ptr(), env._stream()),
                       "pcgrl_step")
            step_no[0] += 1
            e1.record()
            evs.append(("k", e0, e1))
            env._after_step()     # auto-reset launches (inside the timed region)
        t1.record()
        torch.cuda.synchronize()
        kern = sum(x.elapsed_time(y) for tag, x, y in evs if tag == "k")
        flush_ms = sum(x.elapsed_time(y) for tag, x, y in evs if tag == "f")
        return kern, t0.elapsed_time(t1) - flush_ms

    # ---- device-resident arm -----------------------------------------------------------------
    run_steps(warmup)
    barrier()
    if clock_sampler is not None:
        clock_sampler.start()
    launches0 = lib.pcgrl_launch_count()
    kern_ms, region_ms = run_steps(steps)
    launches = lib.pcgrl_launch_count() - launches0
    barrier()
    clocks = clock_sampler.stop() if clock_sampler is not None else None
    t = torch.tensor([region_ms, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    region_ms, kern_ms = float(t[0]), float(t[1])
    value = world * n_envs * steps / (region_ms * 1e-3)
    if dump_dir is not None and rank == 0:
        dump_outputs(env, dump_dir)

    # ---- end-to-end arm (host buffers through the public API) -----------------------------------
    e2e = None
    if not a.no_e2e:
        rng = np.random.default_rng(a.seed + 100 + rank)
        k_e2e = min(steps, e2e_steps)      # never more timed steps than the device-resident arm was given
        HP = min(k_e2e + 3, max(8, int(2e9 // bytes_a)))
        if rep == "cellular":
            host_acts = [act_pool[i % POOL].cpu().pin_memory() for i in range(HP)]
        else:
            host_acts = []
            for _ in range(HP):
                buf = env.host_action_buffer(None)
                buf.view(torch.uint8).numpy().view(dt_a).reshape(shape_a)[...] = rng.integers(0, n_act, size=shape_a).astype(dt_a)
                host_acts.append(buf)
        for i in range(3):
            env.step_host(host_acts[i % HP])
        barrier()
        w0 = time.perf_counter()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        sink = 0.0
        fl = []
        for i in range(k_e2e):
            if flush is not None:      # the L2 flush of small shards is not part of a step: timed, then taken out
                f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
                f0.record(); flush.fill_(i & 0xFF); f1.record()
                fl.append((f0, f1))
            r, d, s = env.step_host(host_acts[(i + 3) % HP])
            sink += float(r[0]) + float(s[0, 0]) + float(d[0])
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - w0
        flush_s = sum(x.elapsed_time(y) for x, y in fl) * 1e-3      # step_host waits for it: it is serial with the step
        te = torch.tensor([max(e0.elapsed_time(e1) * 1e-3, wall) - flush_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        h2d, d2h = env.host_io_bytes()
        api = ("BatchedPcgrlEnv(compact_host_io=True).step_host -> pcgrl_step_host_packed (pinned %s actions H2D; ONE "
               "packed record array D2H: reward f32 | stats %s | done | changed, %d B per env; sync; binary / zelda "
               "shards pipelined in chunks over 3 compute streams + an upload and a download stream)" % (np.dtype(dt_a).name, env.record_dtype()["stats"].base.name,
                                                               env.record_stride)) if env.compact_host_io else \
              ("BatchedPcgrlEnv.step_host -> pcgrl_step_host (pinned int32 actions H2D; reward, done, int32 stats D2H to "
               "pinned host buffers; sync; binary / zelda shards pipelined in chunks over 3 compute streams + an upload and a download stream)")
        e2e = {"value": world * n_envs * k_e2e / float(te[0]), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": k_e2e, "api": api}

    # ---- roofline of the dominant kernel ------------------------------------------------------------
    peak, peak_src = peaks()
    step_bytes = env.step_bytes()
    per_launch_ms = kern_ms / steps
    achieved = step_bytes * n_envs / (per_launch_ms * 1e-3) / 1e9
    if env.cache is not None:      # binary with the incremental search (csrc/step_split.cu), path by shard size
        kernel = "k_split_act + k_split_stats_inc + k_split_out" if n_envs >= (224 << 10) else \
            "k_step_inc" if n_envs >= (24 << 10) else "k_step_lanegroup"
    elif problem in ("binary", "zelda", "binary_holey"):
        kernel = "k_step_bitboard"
    elif problem == "sokoban":
        kernel = "k_step_search<SokobanProb> + k_sokoban_solve + k_sokoban_astar + k_sokoban_combine"
    elif problem == "smb":
        kernel = "k_step_search<SmbProb> + k_smb_solve + k_smb_fallback"
    else:
        kernel = "k_step_search"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "kernel": kernel, "algorithmic_bytes_per_env_step": step_bytes,
                "kernel_ms_per_launch": per_launch_ms, "peak_source": peak_src,
                "note": "HBM bound is loose for this path; the binding resource is SM issue (see profiles/)"}
    prof = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(prof):
        try:
            with open(prof) as f:
                roofline["traffic"] = json.load(f).get(workload)
        except Exception:  # noqa: BLE001
            pass
    from control_pcgrl_b200.dist import reduce_episode_stats
    red = reduce_episode_stats(env.stats, names=env.stat_names)   # the one optional collective, off the step path
    out = {"value": value, "ms_per_step": region_ms / steps, "steps": steps, "warmup": warmup,
           "envs_per_gpu": n_envs, "global_envs": world * n_envs, "e2e": e2e, "roofline": roofline,
           "gpu_launches": int(launches), "clocks": clocks, "pool": POOL,
           "episode_steps": int(env.max_iterations) + 1,
           "l2": ("inputs larger than L2 (%.0f MB grids)" % (grid_bytes / 1e6)) if flush is None
                 else "256 MB L2 flush between steps (excluded from the timing)",
           "action_dtype": np.dtype(dt_a).name,
           "mean_stats": {n: float(v) for n, v in zip(env.stat_names, red["mean"].tolist())}}
    del env, act_all, act_pool, flush
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------- main
def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    problem, rep, shape, obs_window, controls, default_envs = WORKLOADS[a.workload]
    n_envs = a.envs or default_envs
    cores_avail = len(os.sched_getaffinity(0))
    secondary = [] if (a.no_configs or a.workload != "binary-narrow-16x16" or a.envs) else SECONDARY

    if a.impl == "reference":
        if rank != 0:
            return
        seconds = max(2.0, min(20.0, 0.02 * (a.steps + a.warmup)))
        rate, kind, cores, sample = cpu_arm(a.workload, seconds, cores_avail, a.seed)
        configs = {}
        for wl, *_ in secondary:
            r2, k2, c2, s2 = cpu_arm(wl, 3.0, cores_avail, a.seed)
            configs[wl] = {"value": r2, "unit": UNIT, "cpu_baseline": {"value": r2, "unit": UNIT, "cores": c2,
                                                                       "kind": k2, "sample": s2}}
        line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int8/int32 stats, f64 reward", "data": "synthetic",
                "config": {"workload": a.workload, "envs_per_gpu": n_envs},
                "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
                "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "configs": configs}
        print(json.dumps(line), flush=True)
        return

    import torch
    import torch.distributed as dist
    from control_pcgrl_b200 import _lib
    from control_pcgrl_b200.dist import bind_to_gpu_cpus, init_from_env

    if world > 1:
        init_from_env("nccl")
    torch.cuda.set_device(local)
    _lib.load()
    # one process per GPU: stay on the host cores / NUMA node local to this GPU (pinned buffers follow)
    bound = bind_to_gpu_cpus(local) if world > 1 else []

    head = run_workload(a, a.workload, n_envs, a.steps, a.warmup, 200, rank, world, local,
                        clock_sampler=ClockSampler(local) if rank == 0 else None, dump_dir=a.dump_outputs)
    configs = {}
    for wl, envs2, steps2, warm2, e2e2 in secondary:
        try:
            res = run_workload(a, wl, envs2, steps2, warm2, e2e2, rank, world, local)
        except Exception as exc:  # noqa: BLE001 -- a secondary config must not take the headline line down
            res = {"error": f"{type(exc).__name__}: {exc}"}
        configs[wl] = res

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu = None
    if not a.no_cpu_baseline:
        rate, kind, cores, sample = cpu_arm(a.workload, a.cpu_seconds, 1, a.seed)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
               "host_cores_available": cores_avail}
        if world == 1:
            for wl in configs:
                if "error" in configs[wl]:
                    continue
                r2, k2, c2, s2 = cpu_arm(wl, 3.0, 1, a.seed)
                configs[wl]["cpu_baseline"] = {"value": r2, "unit": UNIT, "cores": c2, "kind": k2, "sample": s2}
    for wl, res in configs.items():
        res["metric"], res["unit"] = METRIC, UNIT

    line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int8 grids / int32 stats / f64 reward math", "data": "synthetic",
            "config": {"workload": a.workload, "envs_per_gpu": n_envs, "global_envs": world * n_envs,
                       "actions": f"uniform random {head['action_dtype']}, {head['pool']} distinct pre-generated batches "
                                  "resident in HBM",
                       "episode_steps": head["episode_steps"], "auto_reset": True, "l2": head["l2"],
                       "parallelism": f"env-sharded x{world}, no collective on the step path",
                       "host_cores_bound_rank0": len(bound)},
            "roofline": head["roofline"], "cpu_baseline": cpu, "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
            "clocks": head["clocks"], "mean_stats": head["mean_stats"], "configs": configs}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
