"""Reference for amira_gmg_correct_bubble_reads: a plain loop that restates its definition (include/amira_gmg.h) over
the exported arrays `a`, unitig_loop's output `u`, bubble_loop's output `bub` and the encoded reads, and the test
double with DeviceGraph.correct_bubble_reads built on it.  correct_loop walks every read window by window and finds
each edit as a run of windows across a whole branch by positions (one unitig, one orientation, the position moving by
one); it does not use the read steps, and it asserts that the edits of a read do not overlap.  TEST INFRASTRUCTURE
ONLY."""
from fractions import Fraction

import numpy as np

from tests.bubble_reference import BubbleDevice, bubble_loop
from tests.unitig_path_reference import read_path_loop
from tests.unitig_reference import unitig_loop


def check_replace_with(bub, replace_with):
    off = bub["branch_off"].tolist()
    NB = off[-1]
    if len(replace_with) != NB:
        raise ValueError("replace_with has %d entries for %d branches" % (len(replace_with), NB))
    for b in range(len(off) - 1):
        for g in range(off[b], off[b + 1]):
            x = int(replace_with[g])
            if x != -1 and not (off[b] <= x < off[b + 1] and x != g):
                raise ValueError("replace_with[%d] = %d" % (g, x))


def correct_loop(a, u, bub, ids, off, ps, pe, replace_with):
    """per read: the windows i with a whole branch g (replace_with[g] >= 0) run over windows i .. i + m - 1, live
    windows i - 1 and i + m on the states (sigma, tau) or (tau ^ 1, sigma ^ 1); each such edit replaces calls
    [i, i + m) by the first genes of the kept branch's nodes in the direction of travel"""
    check_replace_with(bub, replace_with)
    woff, wn, wd = a["win_off"].tolist(), a["win_node"].tolist(), a["win_dir"].tolist()
    key = a["node_key"].tolist()
    nu, npos, no = u["node_unitig"].tolist(), u["node_pos"].tolist(), u["node_orient"].tolist()
    uoff, unodes = u["unitig_off"].tolist(), u["unitig_nodes"].tolist()
    boff, bun, bor = bub["branch_off"].tolist(), bub["branch_unitig"].tolist(), bub["branch_orient"].tolist()
    source, sink = bub["source"].tolist(), bub["sink"].tolist()
    branch_of, bubble_of = {}, {}
    for q in range(len(boff) - 1):
        for g in range(boff[q], boff[q + 1]):
            branch_of[bun[g]] = g
            bubble_of[g] = q
    ids, off = np.asarray(ids).tolist(), np.asarray(off).tolist()
    ps = None if ps is None else np.asarray(ps).tolist()
    pe = None if pe is None else np.asarray(pe).tolist()

    def state(w):
        return 2 * wn[w] + (1 if wd[w] < 0 else 0)

    out_ids, out_ps, out_pe, new_off = [], [], [], [0]
    changed, rewritten = [0] * (len(off) - 1), [0] * len(bun)
    for r in range(len(off) - 1):
        w0, nw = woff[r], woff[r + 1] - woff[r]
        edits = []                                             # (first window, m, genes)
        for i in range(1, nw):
            n = wn[w0 + i]
            if n < 0 or nu[n] not in branch_of:
                continue
            b = nu[n]
            g = branch_of[b]
            keep = int(replace_with[g])
            m = uoff[b + 1] - uoff[b]
            if keep < 0 or i + m >= nw:
                continue
            o = wd[w0 + i] * no[n]
            run = all(wn[w0 + i + j] >= 0 and nu[wn[w0 + i + j]] == b and wd[w0 + i + j] * no[wn[w0 + i + j]] == o
                      and npos[wn[w0 + i + j]] == npos[n] + o * j for j in range(m))
            if not run or wn[w0 + i - 1] < 0 or wn[w0 + i + m] < 0:
                continue
            sp, sn = state(w0 + i - 1), state(w0 + i + m)
            sigma, tau = source[bubble_of[g]], sink[bubble_of[g]]
            if (sp, sn) == (sigma, tau):
                travel = 1
            elif (sp, sn) == (tau ^ 1, sigma ^ 1):
                travel = -1
            else:
                continue
            kb = bun[keep]
            walk = travel * bor[keep]
            nodes = unodes[uoff[kb]:uoff[kb + 1]]
            if walk < 0:
                nodes = nodes[::-1]
            genes = [key[x][0] if walk * no[x] > 0 else -key[x][-1] for x in nodes]
            edits.append((i, m, genes))
            rewritten[g] += 1
        for (i1, m1, _), (i2, _, _) in zip(edits, edits[1:]):
            assert i2 >= i1 + m1 + 1, ("edits overlap", r, i1, m1, i2)
        c = off[r]
        for i, m, genes in edits:
            c0 = off[r] + i
            out_ids.extend(ids[c:c0])
            out_ids.extend(genes)
            for src, dst in ((ps, out_ps), (pe, out_pe)):
                if src is not None:
                    dst.extend(src[c:c0])
                    dst.extend(src[c0 + min(j, m - 1)] for j in range(len(genes)))
            c = c0 + m
        out_ids.extend(ids[c:off[r + 1]])
        for src, dst in ((ps, out_ps), (pe, out_pe)):
            if src is not None:
                dst.extend(src[c:off[r + 1]])
        changed[r] = 1 if edits else 0
        new_off.append(len(out_ids))
    return {"ids": np.asarray(out_ids, np.int32), "off": np.asarray(new_off, np.int64),
            "pos_start": None if ps is None else np.asarray(out_ps, np.int32),
            "pos_end": None if pe is None else np.asarray(out_pe, np.int32),
            "changed": np.asarray(changed, np.uint8), "branch_rewritten": np.asarray(rewritten, np.uint32)}


class CorrectionDevice(BubbleDevice):
    """the test double with correct_bubble_reads: correct_loop over the oracle's arrays and the CSR it was built from"""

    def build(self, ids, off, k, pos_start=None, pos_end=None, on_device=False):
        self._csr = tuple(None if x is None else np.asarray(x).copy() for x in (ids, off, pos_start, pos_end))
        return super().build(ids, off, k, pos_start, pos_end, on_device)

    def correct_bubble_reads(self, replace_with, on_device=False):
        a = self.arrays()
        u = unitig_loop(a)
        return correct_loop(a, u, bubble_loop(a, u, read_path_loop(a, u)), *self._csr, np.asarray(replace_with))


def replace_loop(u, bub, amr):
    """replace_with of correct_compacted_bubbles: per bubble the branch with the largest mean node coverage (ties: most
    branch_reads, then the first) replaces every other branch without a node in amr"""
    uoff, unodes, cov_sum = u["unitig_off"].tolist(), u["unitig_nodes"].tolist(), u["cov_sum"].tolist()
    off, bu, rd = bub["branch_off"].tolist(), bub["branch_unitig"].tolist(), bub["branch_reads"].tolist()
    out = [-1] * len(bu)
    for i in range(len(off) - 1):
        best = max(range(off[i], off[i + 1]),
                   key=lambda g: (Fraction(cov_sum[bu[g]], uoff[bu[g] + 1] - uoff[bu[g]]), rd[g], -g))
        for g in range(off[i], off[i + 1]):
            if g != best and not any(amr[n] for n in unodes[uoff[bu[g]]:uoff[bu[g] + 1]]):
                out[g] = best
    return np.asarray(out, np.int64)
