#!/usr/bin/env python
"""Device-time the level-distance kernels (level_knn, level_diversity) against the torch workaround they replace: a
one-hot matmul in bf16 with float32 output (distance = cells - matches), torch.topk per chunk and a merge of the chunks'
candidates; for diversity one batched matmul per group.

    python scripts/bench_level_distance.py [--reps R] [--out profiles/r03_level_distance.jsonl]

Workloads (random levels, every tile code equally likely; both sides read the same tensors):
  (a) 64 Ki binary 16x16 queries against a 1 Mi archive, k = 15
  (b) 1 Ki queries against the same archive (the archive is split into slices and merged)
  (c) diversity of 1 Mi binary levels in groups of 16, and of 64 Ki zelda 7x11 levels in groups of 16
  (d) 16 Ki minecraft_3D_maze 14^3 queries against a 64 Ki archive, k = 10
The workaround's distance chunks are at most 4 GiB of float32.  Times come from CUDA events (R calls of the kernel path,
one of the workaround after one warm-up).  Each workaround result is checked against the kernel's: kNN distances must be
equal, and every workaround index must point at a level of the claimed distance (torch.topk orders ties arbitrarily, so
the index sets agree only where no tie crosses the k-th distance; their agreement is reported); diversity sums must be
equal.  Every line carries the GPU name and power limit read in the same run.
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
from control_pcgrl_b200.problems import get_spec  # noqa: E402

DEV = "cuda:0"
CHUNK_BYTES = 4 << 30


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power}


def events_ms(fn, reps, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def levels(n, problem, shape, seed):
    cells = 1
    for d in shape:
        cells *= d
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(0, get_spec(problem, shape).n_tiles, (n, cells), generator=g, device=DEV,
                         dtype=torch.int32).to(torch.int8)


def onehot(a, n_tiles):
    return torch.nn.functional.one_hot(a.long(), n_tiles).flatten(1).to(torch.bfloat16)


def torch_knn(q, b, k, n_tiles):
    """Chunked one-hot matmul + topk per chunk + a merge; distances exact (counts <= 2^24 in float32)."""
    cells = q.shape[1]
    ob = onehot(b, n_tiles)
    cb = min(b.shape[0], max(1, CHUNK_BYTES // 4 // min(q.shape[0], 4096)))
    cq = max(1, min(q.shape[0], CHUNK_BYTES // 4 // cb))
    dist = torch.empty((q.shape[0], k), dtype=torch.int32, device=DEV)
    idx = torch.empty((q.shape[0], k), dtype=torch.int64, device=DEV)
    for lo in range(0, q.shape[0], cq):
        oq = onehot(q[lo:lo + cq], n_tiles)
        cand_d, cand_i = [], []
        for blo in range(0, b.shape[0], cb):
            d = cells - torch.mm(oq, ob[blo:blo + cb].T, out_dtype=torch.float32)
            v, i = torch.topk(d, min(k, d.shape[1]), dim=1, largest=False)
            cand_d.append(v)
            cand_i.append(i + blo)
        v, j = torch.topk(torch.cat(cand_d, 1), k, dim=1, largest=False)
        dist[lo:lo + cq] = v.to(torch.int32)
        idx[lo:lo + cq] = torch.cat(cand_i, 1).gather(1, j)
    return dist, idx


def torch_div(a, s, n_tiles):
    o = onehot(a, n_tiles).view(a.shape[0] // s, s, -1)
    m = torch.bmm(o, o.transpose(1, 2), out_dtype=torch.float32)
    d = a.shape[1] - m
    return torch.triu(d, diagonal=1).sum((1, 2)).to(torch.int64)


def check_knn(q, b, got, ref):
    d_ok = torch.equal(got[0], ref[0])
    a = torch.sort(got[1].long(), 1).values
    r = torch.sort(ref[1], 1).values
    rows = torch.arange(q.shape[0], device=DEV)[:4096]
    dd = (q[rows, None, :] != b[ref[1][rows]]).sum(-1).to(torch.int32)   # the workaround's indices, recomputed
    return {"dist_equal": bool(d_ok), "ref_idx_consistent_first_4096": bool(torch.equal(dd, ref[0][rows])),
            "idx_sets_equal_frac": float((a == r).all(1).float().mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_level_distance.jsonl"))
    ap.add_argument("--scale", type=int, default=1, help="divide every count by this (a quick rehearsal)")
    args = ap.parse_args()
    info = gpu_info()
    S = args.scale
    lines = []
    binary = P.make_config("binary", "narrow", map_shape=(16, 16))
    arch = levels((1 << 20) // S, "binary", (16, 16), 1)
    for label, nq in (("(a) knn binary 16x16, 64 Ki x 1 Mi, k=15", (1 << 16) // S),
                      ("(b) knn binary 16x16, 1 Ki x 1 Mi, k=15", 1024 // S)):
        q = levels(nq, "binary", (16, 16), 2)
        t, got = events_ms(lambda: P.level_knn(q, arch, k=15, cfg=binary), args.reps)
        tw, ref = events_ms(lambda: torch_knn(q, arch, 15, 2), 1)
        pairs = nq * arch.shape[0]
        lines.append(dict(workload=label, n_query=nq, n_archive=arch.shape[0], k=15, kernel_ms=t, torch_ms=tw,
                          pairs_per_s=pairs / t * 1e3, torch_pairs_per_s=pairs / tw * 1e3, speedup=tw / t,
                          **check_knn(q, arch, got, ref)))
    for label, problem, shape, n in (("(c) diversity binary 16x16, 1 Mi in groups of 16", "binary", (16, 16), 1 << 20),
                                     ("(c) diversity zelda 7x11, 64 Ki in groups of 16", "zelda", (7, 11), 1 << 16)):
        cfg = P.make_config(problem, "narrow", map_shape=shape)
        a = levels(n // S, problem, shape, 3)
        sz = len(a) // 16 * 16
        a = a[:sz]
        t, got = events_ms(lambda: P.level_diversity(a, 16, cfg=cfg), args.reps)
        tw, ref = events_ms(lambda: torch_div(a, 16, get_spec(problem, shape).n_tiles), 1)
        pairs = sz // 16 * 120
        lines.append(dict(workload=label, n_levels=sz, group_size=16, kernel_ms=t, torch_ms=tw,
                          pairs_per_s=pairs / t * 1e3, torch_pairs_per_s=pairs / tw * 1e3, speedup=tw / t,
                          sums_equal=bool(torch.equal(torch.round(got * 120).to(torch.int64), ref))))
    mc = P.make_config("minecraft_3D_maze", "narrow", map_shape=(14, 14, 14))
    q = levels((1 << 14) // S, "minecraft_3D_maze", (14, 14, 14), 4)
    b = levels((1 << 16) // S, "minecraft_3D_maze", (14, 14, 14), 5)
    t, got = events_ms(lambda: P.level_knn(q, b, k=10, cfg=mc), args.reps)
    tw, ref = events_ms(lambda: torch_knn(q, b, 10, get_spec("minecraft_3D_maze", (14, 14, 14)).n_tiles), 1)
    pairs = q.shape[0] * b.shape[0]
    lines.append(dict(workload="(d) knn minecraft_3D_maze 14^3, 16 Ki x 64 Ki, k=10", n_query=q.shape[0],
                      n_archive=b.shape[0], k=10, kernel_ms=t, torch_ms=tw, pairs_per_s=pairs / t * 1e3,
                      torch_pairs_per_s=pairs / tw * 1e3, speedup=tw / t, **check_knn(q, b, got, ref)))
    with open(args.out, "w") as f:
        for ln in lines:
            ln.update(info)
            print(json.dumps(ln), flush=True)
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
