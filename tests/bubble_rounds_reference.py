"""Reference for GeneMerGraph.correct_bubbles_until_stable and amira_gmg_bubble_policy: PolicyDevice, the test double
with DeviceGraph.bubble_policy / bubble_counts built on replace_loop (tests/bubble_correction_reference.py), and
rounds_loop, the composition of existing methods that defines correct_bubbles_until_stable (correct_compacted_bubbles,
a rebuild from its reads, the filter), with the per round counts taken from replace_loop.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

from amira_b200 import _lib, construct_graph
from tests.bubble_correction_reference import CorrectionDevice, replace_loop
from tests.bubble_reference import bubble_loop
from tests.unitig_path_reference import read_path_loop
from tests.unitig_reference import unitig_loop


def spared_nodes(a, ranks):
    """per node: it holds a gene of the ranks (amira_gmg_nodes_containing)"""
    key = np.abs(np.asarray(a["node_key"], np.int64))
    return np.isin(key, list(ranks)).any(axis=1) if len(ranks) and len(key) else np.zeros(len(a["node_cov"]), bool)


class PolicyDevice(CorrectionDevice):
    """the test double with bubble_policy: replace_loop over the oracle's arrays, kept for correct_bubble_reads(None)
    until the graph changes"""
    _policy = None

    def build(self, ids, off, k, pos_start=None, pos_end=None, on_device=False):
        self._policy = None
        return super().build(ids, off, k, pos_start, pos_end, on_device)

    def _with_masks(self, op):
        self._policy = None
        return super()._with_masks(op)

    def bubble_counts(self):
        bub = self.bubbles()
        return len(bub["source"]), len(bub["branch_unitig"])

    def bubble_policy(self, spare_ranks=(), want_replace_with=False):
        a = self.arrays()
        u = unitig_loop(a)
        rw = replace_loop(u, bubble_loop(a, u, read_path_loop(a, u)), spared_nodes(a, spare_ranks))
        self._policy = rw
        n = int((rw >= 0).sum())
        return (n, rw.astype(np.int32)) if want_replace_with else n

    def correct_bubble_reads(self, replace_with=None, on_device=False, flags_on_device=False):
        if replace_with is None:
            if self._policy is None and self.bubble_counts()[1]:
                raise _lib.AmiraLibraryError("amira_gmg status %d: no bubble policy" % _lib.E_STATE)
            replace_with = self._policy if self._policy is not None else np.zeros(0, np.int64)
        else:
            self._policy = None
        return super().correct_bubble_reads(replace_with)


def reference_policy(g, genes):
    """(bubbles, replace_with) of graph g by the reference loops: a lazy graph's device arrays, or a host-edited
    graph's objects"""
    if g._on_device():
        a = w = g._require_device_state().arrays()
        amr = spared_nodes(a, g._gene_ranks(list(genes)))
    else:
        a, w = g._unitig_index_arrays(), g._read_index_arrays()
        amr_nodes = g.get_AMR_nodes(genes)
        amr = np.asarray([nh in amr_nodes for nh in g._nodes], bool)
    u = unitig_loop(a)
    bub = bubble_loop(a, u, read_path_loop({**a, **w}, u))
    return bub, replace_loop(u, bub, amr)


def round_counts(g, genes, fast=False):
    """bubbles, branches and branches replaced of graph g; fast: the bubbles and unitigs from the graph's own (tested)
    compacted_bubbles / compacted_unitigs, for inputs too large for the loops"""
    if fast:
        bub, u = g.compacted_bubbles(), g.compacted_unitigs()
        if g._on_device():
            amr = spared_nodes(g._require_device_state().arrays(), g._gene_ranks(list(genes)))
        else:
            amr_nodes = g.get_AMR_nodes(genes)
            amr = np.asarray([nh in amr_nodes for nh in g._nodes], bool)
        rw = replace_loop(u, bub, amr)
    else:
        bub, rw = reference_policy(g, genes)
    return {"bubbles": len(bub["source"]), "branches": len(bub["branch_unitig"]), "replaced": int((rw >= 0).sum())}


def rounds_loop(g, max_rounds=30, genes={}, filter_graph=None, fast=False):
    """correct_bubbles_until_stable by its definition -> (graph, reads, changed union, rounds)"""
    cur, e = g, g._source_encoded()
    changed, rounds = np.zeros(len(e.read_ids), np.uint8), []
    for _ in range(max_rounds):
        counts = round_counts(cur, genes, fast)
        e2 = cur.correct_compacted_bubbles(genes)
        rounds.append({**counts, "steps": int(e2.branch_rewritten.sum()), "reads": int(e2.changed.sum()),
                       "calls": len(e2.ids)})
        if not e2.branch_rewritten.any():
            break
        e, changed = e2, changed | e2.changed
        cur = construct_graph.GeneMerGraph(e, g._kmerSize)
        if filter_graph:
            cur.filter_graph(*filter_graph)
    return cur, e, changed, rounds
