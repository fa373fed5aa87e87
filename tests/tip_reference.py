"""Reference for amira_gmg_tips, amira_gmg_tip_policy and amira_gmg_clip_tip_reads: plain loops that restate their
definitions (include/amira_gmg.h) over the exported arrays `a`, unitig_loop's output `u` and read_path_loop's output
`p`, and test doubles with DeviceGraph.tips (TipDevice) and with tip_policy / clip_tip_reads (TipPolicyDevice) built on
them.  tip_loop walks every candidate unitig by positions (node_unitig / node_pos), not through unitig_nodes;
tip_policy_loop compares mean coverages as exact Fractions; clip_loop asserts that the clips of a read do not overlap
and that a clipped read keeps k calls or more.  TEST INFRASTRUCTURE ONLY."""
from fractions import Fraction

import numpy as np

from amira_b200 import _lib
from tests.bubble_rounds_reference import PolicyDevice, spared_nodes
from tests.unitig_path_reference import read_path_loop
from tests.unitig_reference import unitig_loop


def _lists(a):
    fw_off, fw_edges, bw_off, bw_edges = (a[f].tolist() for f in ("fw_off", "fw_edges", "bw_off", "bw_edges"))

    def lst(s):
        n = s >> 1
        return fw_edges[fw_off[n]:fw_off[n + 1]] if s & 1 == 0 else bw_edges[bw_off[n]:bw_off[n + 1]]
    return lst


def tip_loop(a, u, p):
    """unitig by unitig: its nodes in listed order by positions, its two outward end states, and the tip condition"""
    lst = _lists(a)
    tgt, td = a["edge_tgt"].tolist(), a["edge_td"].tolist()
    nu, npos, no = u["node_unitig"].tolist(), u["node_pos"].tolist(), u["node_orient"].tolist()
    circ = u["circular"].tolist()
    members = {}
    for n, b in enumerate(nu):
        members.setdefault(b, []).append(n)
    steps = {}
    for b in p["unitig"].tolist():
        steps[b] = steps.get(b, 0) + 1
    out = {"tip_unitig": [], "tip_orient": [], "tip_attach": [], "tip_reads": []}
    for b in range(len(circ)):
        if circ[b]:
            continue
        nodes = sorted(members[b], key=lambda n: npos[n])
        assert [npos[n] for n in nodes] == list(range(len(nodes)))
        h0, h1 = nodes[0], nodes[-1]
        out1 = 2 * h1 + (1 if no[h1] < 0 else 0)
        out0 = (2 * h0 + (1 if no[h0] < 0 else 0)) ^ 1
        l0, l1 = lst(out0), lst(out1)
        if len(l0) == 0 and len(l1) == 1:
            e, orient = l1[0], -1
        elif len(l1) == 0 and len(l0) == 1:
            e, orient = l0[0], 1
        else:
            continue
        v = tgt[e]
        if nu[v] == b:
            continue
        attach = (2 * v + (1 if td[e] < 0 else 0)) ^ 1
        assert len(lst(attach)) >= 2, ("a tip's junction list holds one edge", b)
        out["tip_unitig"].append(b)
        out["tip_orient"].append(orient)
        out["tip_attach"].append(attach)
        out["tip_reads"].append(steps.get(b, 0))
    return {"tip_unitig": np.asarray(out["tip_unitig"], np.int32), "tip_orient": np.asarray(out["tip_orient"], np.int8),
            "tip_attach": np.asarray(out["tip_attach"], np.int32), "tip_reads": np.asarray(out["tip_reads"], np.uint32)}


def tip_policy_loop(a, u, tips, amr, min_length):
    """per tip: fewer than min_length nodes, no node in amr, and an edge of list(attach) into another unitig whose
    mean node coverage is strictly larger"""
    lst = _lists(a)
    tgt = a["edge_tgt"].tolist()
    nu = u["node_unitig"].tolist()
    uoff, unodes, cov_sum = u["unitig_off"].tolist(), u["unitig_nodes"].tolist(), u["cov_sum"].tolist()

    def mean(c):
        return Fraction(cov_sum[c], uoff[c + 1] - uoff[c])
    out = []
    for b, att in zip(tips["tip_unitig"].tolist(), tips["tip_attach"].tolist()):
        ln = uoff[b + 1] - uoff[b]
        spared = any(amr[n] for n in unodes[uoff[b]:uoff[b + 1]])
        better = any(nu[tgt[e]] != b and mean(nu[tgt[e]]) > mean(b) for e in lst(att))
        out.append(1 if ln < min_length and not spared and better else 0)
    return np.asarray(out, np.uint8)


def clip_loop(a, u, p, tips, ids, off, ps, pe, clip):
    """per read, step by step: an end clip (the step reaches the read's last window from a live window on the attach
    state) drops the last `length` calls, a start clip (the read's first step, followed by a live window on attach ^ 1)
    drops the first `length` calls"""
    clip = np.asarray(clip).ravel()
    if len(clip) != len(tips["tip_unitig"]) or any(int(c) not in (0, 1) for c in clip.tolist()):
        raise ValueError("clip must hold 0 or 1 per tip")
    woff, wn, wd = a["win_off"].tolist(), a["win_node"].tolist(), a["win_dir"].tolist()
    tip_of = {b: q for q, b in enumerate(tips["tip_unitig"].tolist())}
    attach = tips["tip_attach"].tolist()
    path_off, su, sw, sl = (p[f].tolist() for f in ("path_off", "unitig", "win", "length"))
    ids, off = np.asarray(ids).tolist(), np.asarray(off).tolist()
    ps = None if ps is None else np.asarray(ps).tolist()
    pe = None if pe is None else np.asarray(pe).tolist()

    def state(w):
        return 2 * wn[w] + (1 if wd[w] < 0 else 0)

    out_ids, out_ps, out_pe, new_off = [], [], [], [0]
    changed, clipped = [0] * (len(off) - 1), [0] * len(attach)
    for r in range(len(off) - 1):
        w0, nw, nc = woff[r], woff[r + 1] - woff[r], off[r + 1] - off[r]
        lo, hi = 0, nc                                       # the calls kept: [lo, hi)
        for t in range(path_off[r], path_off[r + 1]):
            q = tip_of.get(su[t])
            if q is None or not clip[q]:
                continue
            i, ln = sw[t], sl[t]
            if i >= 1 and i + ln == nw and wn[w0 + i - 1] >= 0 and state(w0 + i - 1) == attach[q]:
                assert hi == nc, ("two end clips", r)
                hi = nc - ln
            elif i == 0 and ln < nw and wn[w0 + ln] >= 0 and state(w0 + ln) == attach[q] ^ 1:
                assert lo == 0, ("two start clips", r)
                lo = ln
            else:
                continue
            clipped[q] += 1
        if (lo, hi) != (0, nc):
            k = nc - nw + 1
            assert lo < hi and hi - lo >= k, ("clips overlap or leave fewer than k calls", r, lo, hi, k)
            changed[r] = 1
        out_ids.extend(ids[off[r] + lo:off[r] + hi])
        for src, dst in ((ps, out_ps), (pe, out_pe)):
            if src is not None:
                dst.extend(src[off[r] + lo:off[r] + hi])
        new_off.append(len(out_ids))
    return {"ids": np.asarray(out_ids, np.int32), "off": np.asarray(new_off, np.int64),
            "pos_start": None if ps is None else np.asarray(out_ps, np.int32),
            "pos_end": None if pe is None else np.asarray(out_pe, np.int32),
            "changed": np.asarray(changed, np.uint8), "tip_clipped": np.asarray(clipped, np.uint32)}


def reference_tips(a):
    """(u, p, tips) of the arrays `a` by the loops"""
    u = unitig_loop(a)
    p = read_path_loop(a, u)
    return u, p, tip_loop(a, u, p)


class TipDevice(PolicyDevice):
    """the test double with tips: tip_loop over the oracle's arrays"""

    def tips(self):
        return reference_tips(self.arrays())[2]


class TipPolicyDevice(TipDevice):
    """the test double with tip_policy / clip_tip_reads: the loops over the oracle's arrays, the policy's flags kept
    for clip_tip_reads(None) until the graph changes"""
    _clip = None

    def build(self, ids, off, k, pos_start=None, pos_end=None, on_device=False):
        self._clip = None
        return super().build(ids, off, k, pos_start, pos_end, on_device)

    def _with_masks(self, op):
        self._clip = None
        return super()._with_masks(op)

    def tip_count(self):
        return len(self.tips()["tip_unitig"])

    def tip_policy(self, min_length, ranks=(), want_clip=False):
        a = self.arrays()
        u, _, tips = reference_tips(a)
        clip = tip_policy_loop(a, u, tips, spared_nodes(a, ranks), min_length)
        self._clip = clip
        return (int(clip.sum()), clip) if want_clip else int(clip.sum())

    def clip_tip_reads(self, clip=None, on_device=False, flags_on_device=False):
        a = self.arrays()
        u, p, tips = reference_tips(a)
        if clip is None:
            if self._clip is None and len(tips["tip_unitig"]):
                raise _lib.AmiraLibraryError("amira_gmg status %d: no tip policy" % _lib.E_STATE)
            clip = self._clip if self._clip is not None else np.zeros(0, np.uint8)
        else:
            self._clip = None
        return clip_loop(a, u, p, tips, *self._csr, clip)
