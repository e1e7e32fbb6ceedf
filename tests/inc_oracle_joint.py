"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the incremental binary search as BinaryIncMachine
(control_pcgrl_b200/csrc/step_split.cu) runs it: the update of oracle/inc_oracle.py `IncBinary.flip`, with two changes
that leave every result and every cache row (P, F, m) as they were.

1. One joint final sweep.  When the edit touches the component that held the old maximum, `IncBinary.flip` sweeps
   twice: from the far tiles of U (inside U), then from the far tiles of the untouched components (outside U).  The
   two regions are different components, so one multi-source BFS from both sets of far tiles gives max(lu, lold) in
   max(lu, lold) levels instead of lu + lold.  Tie rule for m (the old one is `mcu if lu > lold else mold`): the
   lowest cell of (last frontier & untouched region) if that is not empty, else the lowest cell of the last frontier.
2. Local isolated-cell accounting.  Only one cell c changed, so the isolated cells that matter lie next to c.  With
   Q = P' \\ {c} (= P' if c became solid, = P_old if c became passable) and iso(Q) the cells of Q without a neighbour
   in Q:
     c became solid:     old isolated cells in A = {c} if N(c) & Q is empty;  new isolated cells in U = N(c) & iso(Q)
     c became passable:  old isolated cells in A = N(c) & iso(Q);             new isolated cells in U = {c} if N(c) & Q
                                                                                                       is empty
   (U is connected from c or from c's neighbours: a cell of U without a neighbour in P_old, or in P', can only touch
   the rest of U through c.)
"""
from __future__ import annotations

from oracle.inc_oracle import IncBinary


def popcount(s):
    return bin(s).count("1")


class IncBinaryJoint(IncBinary):
    def flip(self, y, x):
        """The cell (y, x) changes passability.  Same results and cache as IncBinary.flip."""
        c = 1 << (y * self.W + x)
        Po, Pn = self.P, self.P ^ c
        grew = bool(Pn & c)
        q = Pn & ~c                                                      # Q: P' without c
        nc = self.nbr(c) & q                                             # c's passable neighbours
        iso_nb = nc & ~self.nbr(q)                                       # ... that have no other neighbour
        c_alone = c if not nc else 0
        seed = c if grew else nc
        _, _, U = self.bfs(seed, Pn & ~seed) if seed else (0, 0, 0)    # every NEW component the edit affects
        A = U | (0 if grew else c)                                       # covers every affected OLD component
        iso_old, iso_new = (iso_nb, c_alone) if grew else (c_alone, iso_nb)
        k_old = popcount(self.F & A) + popcount(iso_old)
        f_rest = self.F & ~A                                             # far tiles of the untouched components
        hit = self.m >= 0 and (A >> self.m) & 1
        regions = self.regions - k_old + popcount(iso_new)
        avail, fars = U & ~iso_new, 0
        while avail:                                                     # first sweeps inside U
            s = self.lowest(avail)
            _, last, reached = self.bfs(s, avail & ~s)
            fars |= self.lowest(last)
            avail &= ~reached
            regions += 1
        src = fars | (f_rest if hit else 0)                              # joint final sweep
        if src:
            path, last, _ = self.bfs(src, Pn & ~src)
        else:
            path, last = 0, 0
        if hit:
            rest = last & ~U                                             # untouched components win ties
            m = self.lowest(rest or last).bit_length() - 1
        elif path > self.path:
            m = self.lowest(last).bit_length() - 1
        else:
            path, m = self.path, self.m
        self.P, self.F, self.regions, self.path, self.m = Pn, f_rest | fars, regions, path, m
        return self.regions, self.path
