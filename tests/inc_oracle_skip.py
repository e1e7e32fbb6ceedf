"""TEST INFRASTRUCTURE ONLY -- CPU restatement of BinaryIncMachine (control_pcgrl_b200/csrc/step_split.cu) with the
skipped final sweep: tests/inc_oracle_joint.py's update, which leaves every result and every cache row (P, F, m) as it
was, plus one rule that proves the final sweep useless before running it.

When the edit does not touch the component that held the old maximum (`hit` false), the final sweep runs from the far
tiles of U only and can only raise path-length: path' = max(path, lu), with lu the largest eccentricity of a far tile
of U.  The first sweep of component C_j of U from its first tile reaches depth e1_j = ecc(first_j), so

    ecc(far_j) <= d(far_j, first_j) + ecc(first_j) = 2 * e1_j.

If max_j 2 * e1_j <= path, then lu <= path: path and m stay as they are (a tie keeps the old m, as in the joint
update), so the sweep is not run.  The regions count and the new far tiles come from the first sweeps.
"""
from __future__ import annotations

from tests.inc_oracle_joint import IncBinaryJoint, popcount


class IncBinarySkip(IncBinaryJoint):
    """Same results and cache as IncBinaryJoint.flip.  `skipped` counts the edits whose final sweep was skipped."""
    skipped = 0

    def flip(self, y, x):
        c = 1 << (y * self.W + x)
        Pn = self.P ^ c
        grew = bool(Pn & c)
        q = Pn & ~c
        nc = self.nbr(c) & q
        iso_nb = nc & ~self.nbr(q)
        c_alone = c if not nc else 0
        seed = c if grew else nc
        _, _, U = self.bfs(seed, Pn & ~seed) if seed else (0, 0, 0)
        A = U | (0 if grew else c)
        iso_old, iso_new = (iso_nb, c_alone) if grew else (c_alone, iso_nb)
        k_old = popcount(self.F & A) + popcount(iso_old)
        f_rest = self.F & ~A
        hit = self.m >= 0 and (A >> self.m) & 1
        regions = self.regions - k_old + popcount(iso_new)
        avail, fars, e1_max = U & ~iso_new, 0, 0
        while avail:                                                     # first sweeps inside U
            s = self.lowest(avail)
            e1, last, reached = self.bfs(s, avail & ~s)
            fars |= self.lowest(last)
            avail &= ~reached
            regions += 1
            e1_max = max(e1_max, e1)
        if not hit and 2 * e1_max <= self.path:                          # the final sweep cannot change path or m
            self.skipped += 1
            self.P, self.F, self.regions = Pn, f_rest | fars, regions
            return self.regions, self.path
        src = fars | (f_rest if hit else 0)                              # joint final sweep
        if src:
            path, last, _ = self.bfs(src, Pn & ~src)
        else:
            path, last = 0, 0
        if hit:
            rest = last & ~U
            m = self.lowest(rest or last).bit_length() - 1
        elif path > self.path:
            m = self.lowest(last).bit_length() - 1
        else:
            path, m = self.path, self.m
        self.P, self.F, self.regions, self.path, self.m = Pn, f_rest | fars, regions, path, m
        return self.regions, self.path
