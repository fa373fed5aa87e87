"""Reference for amira_gmg_clean_reads and GeneMerGraph.clean_until_stable: clean_loop composes the two committed
loops, correct_loop (tests/bubble_correction_reference.py) and clip_loop (tests/tip_reference.py), on one graph;
CleanDevice is the test double with DeviceGraph.clean_reads built on it; clean_rounds_loop is the composition of
existing methods that defines clean_until_stable, with the per round counts taken from the loops.  TEST
INFRASTRUCTURE ONLY."""
import numpy as np

from amira_b200 import _lib, construct_graph
from tests.bubble_correction_reference import check_replace_with, correct_loop, replace_loop
from tests.bubble_reference import bubble_loop
from tests.bubble_rounds_reference import spared_nodes
from tests.tip_reference import TipPolicyDevice, clip_loop, reference_tips, tip_loop, tip_policy_loop
from tests.unitig_path_reference import read_path_loop
from tests.unitig_reference import unitig_loop

MARK = 1 << 30          # call c of the input travels through the loops as the id MARK + c; no gene id reaches it


def clean_loop(a, u, bub, p, tips, ids, off, ps, pe, replace_with, clip):
    """per read: the bubble-corrected read of correct_loop minus the calls clip_loop drops at its two ends, positions
    alike.  Both loops run over marked ids, so that the calls the clip drops are known by their input index and the
    calls of the corrected read that are copies of input calls are known too; the dropped calls must be copies,
    untouched by any edit, at the corrected read's two ends"""
    ids, off = np.asarray(ids, np.int64), np.asarray(off, np.int64)
    G, R = len(ids), len(off) - 1
    assert G < MARK
    marked = (MARK + np.arange(G)).astype(np.int32)
    cor = correct_loop(a, u, bub, marked, off, ps, pe, replace_with)
    clp = clip_loop(a, u, p, tips, marked, off, None, None, clip)
    out_ids, out_ps, out_pe, new_off = [], [], [], [0]
    for r in range(R):
        lo_c, hi_c = int(cor["off"][r]), int(cor["off"][r + 1])
        x = cor["ids"][lo_c:hi_c].astype(np.int64)
        kept = clp["ids"][clp["off"][r]:clp["off"][r + 1]].astype(np.int64) - MARK - off[r]
        nc = int(off[r + 1] - off[r])
        head = int(kept[0]) if len(kept) else 0
        tail = nc - head - len(kept)
        assert np.array_equal(kept, np.arange(head, head + len(kept))), ("the clip keeps one run of calls", r)
        assert np.array_equal(x[:head], MARK + off[r] + np.arange(head)), ("a clipped call was edited", r)
        assert np.array_equal(x[len(x) - tail:], MARK + off[r] + np.arange(nc - tail, nc)), ("a clipped call was edited", r)
        y = x[head:len(x) - tail]
        out_ids.extend(np.where(y >= MARK, ids[np.clip(y - MARK, 0, max(G - 1, 0))], y).tolist())
        for src, dst in ((cor["pos_start"], out_ps), (cor["pos_end"], out_pe)):
            if src is not None:
                dst.extend(src[lo_c + head:hi_c - tail].tolist())
        new_off.append(len(out_ids))
    return {"ids": np.asarray(out_ids, np.int32), "off": np.asarray(new_off, np.int64),
            "pos_start": None if ps is None else np.asarray(out_ps, np.int32),
            "pos_end": None if pe is None else np.asarray(out_pe, np.int32),
            "changed": (cor["changed"] | clp["changed"]).astype(np.uint8),
            "branch_rewritten": cor["branch_rewritten"], "tip_clipped": clp["tip_clipped"]}


def check_clip(tips, clip):
    clip = np.asarray(clip).ravel()
    if len(clip) != len(tips["tip_unitig"]) or any(int(c) not in (0, 1) for c in clip.tolist()):
        raise ValueError("clip must hold 0 or 1 per tip")


class CleanDevice(TipPolicyDevice):
    """the test double with clean_reads: clean_loop over the oracle's arrays and the CSR it was built from, with the
    held policies of bubble_policy and tip_policy"""

    def clean_reads(self, replace_with=None, clip=None, on_device=False, flags_on_device=False):
        a = self.arrays()
        u, p, tips = reference_tips(a)
        bub = bubble_loop(a, u, p)
        if replace_with is None and self._policy is None and len(bub["branch_unitig"]):
            raise _lib.AmiraLibraryError("amira_gmg status %d: no bubble policy" % _lib.E_STATE)
        if clip is None and self._clip is None and len(tips["tip_unitig"]):
            raise _lib.AmiraLibraryError("amira_gmg status %d: no tip policy" % _lib.E_STATE)
        if replace_with is not None:
            check_replace_with(bub, np.asarray(replace_with).ravel())
        if clip is not None:
            check_clip(tips, clip)
        if replace_with is None:
            replace_with = self._policy if self._policy is not None else np.zeros(0, np.int64)
        else:
            self._policy = None
        if clip is None:
            clip = self._clip if self._clip is not None else np.zeros(0, np.uint8)
        else:
            self._clip = None
        return clean_loop(a, u, bub, p, tips, *self._csr, np.asarray(replace_with), clip)


def graph_policies(g, genes, min_tip_length, fast=False):
    """(bubbles, replace_with, tips, clip) of graph g: a lazy graph's device arrays or a host-edited graph's objects,
    by the loops; fast: the bubbles, tips and unitigs from the graph's own (tested) compacted_* methods, for inputs
    too large for those loops"""
    if g._on_device():
        a = w = g._require_device_state().arrays()
        amr = spared_nodes(a, g._gene_ranks(list(genes)))
    else:
        a, w = g._unitig_index_arrays(), g._read_index_arrays()
        amr_nodes = g.get_AMR_nodes(genes)
        amr = np.asarray([nh in amr_nodes for nh in g._nodes], bool)
    if fast:
        u, bub, tips = g.compacted_unitigs(), g.compacted_bubbles(), g.compacted_tips()
    else:
        u = unitig_loop(a)
        p = read_path_loop({**a, **w}, u)
        bub, tips = bubble_loop(a, u, p), tip_loop(a, u, p)
    return bub, replace_loop(u, bub, amr), tips, tip_policy_loop(a, u, tips, amr, min_tip_length)


def clean_counts(g, genes, min_tip_length, fast=False):
    bub, rw, tips, clip = graph_policies(g, genes, min_tip_length, fast)
    return {"bubbles": len(bub["source"]), "branches": len(rw), "replaced": int((rw >= 0).sum()),
            "tips": len(clip), "tips_clipped": int(clip.sum())}


def clean_rounds_loop(g, min_tip_length, max_rounds=30, genes={}, filter_graph=None, fast=False):
    """clean_until_stable by its definition -> (graph, reads, changed union, rounds)"""
    cur, e = g, g._source_encoded()
    changed, rounds = np.zeros(len(e.read_ids), np.uint8), []
    for _ in range(max_rounds):
        counts = clean_counts(cur, genes, min_tip_length, fast)
        e2 = cur.clean_compacted_reads(min_tip_length, genes)
        rounds.append({**counts, "steps": int(e2.branch_rewritten.sum()), "steps_clipped": int(e2.tip_clipped.sum()),
                       "reads": int(e2.changed.sum()), "calls": len(e2.ids)})
        if not (e2.branch_rewritten.any() or e2.tip_clipped.any()):
            break
        e, changed = e2, changed | e2.changed
        cur = construct_graph.GeneMerGraph(e, g._kmerSize)
        if filter_graph:
            cur.filter_graph(*filter_graph)
    return cur, e, changed, rounds
