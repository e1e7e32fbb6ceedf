"""Work per changed grid of the incremental binary search, for the two-sweep update (oracle/inc_oracle.py), the
joint-sweep update (tests/inc_oracle_joint.py) and the joint-sweep update with the skipped final sweep that
BinaryIncMachine runs (tests/inc_oracle_skip.py), on 16x16 narrow-representation rollouts (the flagship workload's
edit pattern: the cell cursor walks the map in row-major order, each step sets a random tile).

    segments      BFS runs from a non-empty start (flood, first sweep per component of U, final sweeps)
    expansions    board expansions of those runs, the last (empty) one included
    transitions   calls of the machine's transition step: one per segment, plus one for a flood with no seed

CPU only: counts, not times.  python scripts/inc_work_counts.py [--maps N] [--seed S]"""
import argparse
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle.inc_oracle import IncBinary  # noqa: E402
from tests.inc_oracle_joint import IncBinaryJoint  # noqa: E402
from tests.inc_oracle_skip import IncBinarySkip  # noqa: E402


def counting(cls):
    class Counting(cls):
        segments = expansions = 0

        def bfs(self, front, avail):
            r = cls.bfs(self, front, avail)
            self.segments += 1
            self.expansions += r[0] + 1
            return r
    return Counting


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--maps", type=int, default=120)
    ap.add_argument("--seed", type=int, default=3)
    args = ap.parse_args()
    rng = random.Random(args.seed)
    machines = {"two-sweep": counting(IncBinary), "joint": counting(IncBinaryJoint), "skip": counting(IncBinarySkip)}
    n, no_seed, skipped = 0, 0, 0
    totals = {k: [0, 0] for k in machines}
    for _ in range(args.maps):
        g = [[rng.randrange(2) for _ in range(16)] for _ in range(16)]
        ms = {k: cls(g) for k, cls in machines.items()}
        for m in ms.values():
            m.segments = m.expansions = 0
        s0 = rng.randrange(256)
        for t in range(256):
            y, x = divmod((s0 + t) % 256, 16)
            v = rng.randrange(2)
            if v == g[y][x]:
                continue
            g[y][x] = v
            n += 1
            ref = ms["two-sweep"]
            c = 1 << (y * 16 + x)
            no_seed += bool(ref.P & c) and not (ref.nbr(c) & ref.P)      # became solid with no passable neighbour
            for m in ms.values():
                m.flip(y, x)
        for k, m in ms.items():
            totals[k][0] += m.segments
            totals[k][1] += m.expansions
        skipped += ms["skip"].skipped
        assert len({(m.regions, m.path, m.F, m.m) for m in ms.values()}) == 1
    print(f"{n} changed grids ({args.maps} maps x 256 narrow steps, seed {args.seed})")
    print(f"{'':10s} {'segments':>9s} {'expansions':>11s} {'transitions':>12s}   (per changed grid)")
    for k, (seg, exp) in totals.items():
        print(f"{k:10s} {seg / n:9.2f} {exp / n:11.1f} {(seg + no_seed) / n:12.2f}")
    print(f"final sweep skipped on {skipped / n:.1%} of the changed grids")


if __name__ == "__main__":
    main()
