"""Reference for amira_gmg_bubbles and the popping policy of pop_compacted_bubbles: plain loops that restate their
definitions (include/amira_gmg.h, GeneMerGraph.pop_compacted_bubbles) over the exported arrays `a`, unitig_loop's
output `u` and read_path_loop's output `p`, and the test double with DeviceGraph.bubbles built on them.  bubble_loop
walks every candidate branch by positions (node_unitig / node_pos / node_orient), one node at a time, as
read_path_loop does.  TEST INFRASTRUCTURE ONLY."""
from fractions import Fraction

import numpy as np

from tests.unitig_path_reference import UnitigPathDevice, read_path_loop
from tests.unitig_reference import unitig_loop


def bubble_loop(a, u, p):
    """states in ascending order, list entries in order; each entry that enters a branch is grouped by its tau in
    first-seen order; a group of two or more with sigma < tau ^ 1 is a bubble"""
    fw_off, fw_edges, bw_off, bw_edges = (a[f].tolist() for f in ("fw_off", "fw_edges", "bw_off", "bw_edges"))
    tgt, td = a["edge_tgt"].tolist(), a["edge_td"].tolist()
    nu, npos, no = u["node_unitig"].tolist(), u["node_pos"].tolist(), u["node_orient"].tolist()
    uoff, unodes, circ = u["unitig_off"].tolist(), u["unitig_nodes"].tolist(), u["circular"].tolist()

    def lst(s):
        n = s >> 1
        return fw_edges[fw_off[n]:fw_off[n + 1]] if s & 1 == 0 else bw_edges[bw_off[n]:bw_off[n + 1]]

    def cont(j):
        return 2 * tgt[j] + (1 if td[j] < 0 else 0)

    def branch(sigma, j):
        """(tau, unitig, orientation) of the branch edge j of list(sigma) enters, or None"""
        x, h, c = sigma >> 1, tgt[j], cont(j)
        if len(lst(c ^ 1)) != 1:
            return None
        b = nu[h]
        if circ[b] or nu[x] == b:                             # condition 4 for x first: the walk starts at an end
            return None
        o = 1 if (c & 1) == (1 if no[h] < 0 else 0) else -1    # +1: h is left through its listed state
        size, q, walked = uoff[b + 1] - uoff[b], npos[h], [h]
        while 0 <= q + o < size:
            q += o
            walked.append(unodes[uoff[b] + q])
        assert len(walked) == size, ("branch entered inside its unitig", sigma, j)
        t = walked[-1]
        s_t = 2 * t + ((1 if no[t] < 0 else 0) if o == 1 else (0 if no[t] < 0 else 1))
        out = lst(s_t)
        if len(out) != 1:
            return None
        y = tgt[out[0]]
        if nu[y] == b:
            return None
        return cont(out[0]), b, 1 if unodes[uoff[b]] == h else -1

    source, sink, branch_off, bun, bor = [], [], [0], [], []
    for sigma in range(2 * len(a["node_cov"])):
        groups = {}
        for j in lst(sigma):
            r = branch(sigma, j)
            if r is not None:
                groups.setdefault(r[0], []).append(r[1:])
        for tau, brs in groups.items():
            if len(brs) < 2 or not sigma < (tau ^ 1):
                continue
            source.append(sigma)
            sink.append(tau)
            for b, o in brs:
                bun.append(b)
                bor.append(o)
            branch_off.append(len(bun))
    ulen = np.diff(u["unitig_off"]).tolist()
    full = {}
    for un, ln in zip(p["unitig"].tolist(), p["length"].tolist()):
        if ln == ulen[un]:
            full[un] = full.get(un, 0) + 1
    return {"source": np.asarray(source, np.int32), "sink": np.asarray(sink, np.int32),
            "branch_off": np.asarray(branch_off, np.int64), "branch_unitig": np.asarray(bun, np.int32),
            "branch_orient": np.asarray(bor, np.int8), "branch_reads": np.asarray([full.get(b, 0) for b in bun], np.uint32)}


def pop_loop(u, bub, amr):
    """the node indices pop_compacted_bubbles removes: per bubble the branch with the largest mean node coverage stays
    (ties: most branch_reads, then the first); every other branch goes whole unless a node of it is in amr"""
    uoff, unodes, cov_sum = u["unitig_off"].tolist(), u["unitig_nodes"].tolist(), u["cov_sum"].tolist()
    off, bu, rd = bub["branch_off"].tolist(), bub["branch_unitig"].tolist(), bub["branch_reads"].tolist()
    out = []
    for i in range(len(off) - 1):
        best = None
        for g in range(off[i], off[i + 1]):
            b = bu[g]
            key = (Fraction(cov_sum[b], uoff[b + 1] - uoff[b]), rd[g])
            if best is None or key > best[0]:
                best = (key, g)
        for g in range(off[i], off[i + 1]):
            nodes = unodes[uoff[bu[g]]:uoff[bu[g] + 1]]
            if g != best[1] and not any(amr[n] for n in nodes):
                out.extend(nodes)
    return out


class BubbleDevice(UnitigPathDevice):
    """the test double with bubbles: bubble_loop over the oracle's arrays"""

    def bubbles(self):
        a = self.arrays()
        u = unitig_loop(a)
        return bubble_loop(a, u, read_path_loop(a, u))
