"""Bubble read correction without a GPU: hand-made probes with known answers (a substitution, a deletion and an
insertion at k = 3, a strand flip, a read that crosses the bubble backwards, two bubbles of one read that share a
junction, three branches, a read that starts on the branch, an edge filtered away next to a branch, a branch spared
for a gene of interest, a circle); the rebuild from the corrected reads against the build of the error-free reads; the
product's host implementation (GeneMerGraph._corrected_reads_over) against correct_loop
(tests/bubble_correction_reference.py) on lazy graphs through the test double and on host-edited graphs, after
filters, trimming and remove_node; the positions policy; the source reads left untouched; save / load."""
import copy
import os

import numpy as np
import pytest

from amira_b200 import construct_graph, encode
from oracle import gmg_oracle as O
from tests.bubble_correction_reference import CorrectionDevice, correct_loop, replace_loop
from tests.bubble_reference import bubble_loop
from tests.fake_device import OracleBackedDevice
from tests.test_bubbles_cpu import TRUE, error_reads
from tests.test_unitigs_cpu import FIXTURES
from tests.unitig_path_reference import read_path_loop
from tests.unitig_reference import unitig_loop

ERR_SUB = ["+a", "+b", "+c", "+x", "+e", "+f", "+g"]
ERR_DEL = ["+a", "+b", "+c", "+e", "+f", "+g"]
ERR_INS = ["+a", "+b", "+c", "+x", "+d", "+e", "+f", "+g"]


def rc(read):
    return [("-" if g[0] == "+" else "+") + g[1:] for g in read[::-1]]


@pytest.fixture
def fake_device(monkeypatch):
    """lazy graphs on the test double without the new call: served by the host implementation over its arrays"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", OracleBackedDevice)


@pytest.fixture
def loop_device(monkeypatch):
    """lazy graphs on the test double with the new call, served by correct_loop"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", CorrectionDevice)


def same(x, y, ctx=""):
    assert x.keys() >= {"ids", "off", "pos_start", "pos_end", "changed", "branch_rewritten"}, ctx
    for f in ("ids", "off", "pos_start", "pos_end", "changed", "branch_rewritten"):
        if x[f] is None or y[f] is None:
            assert x[f] is None and y[f] is None, (ctx, f)
            continue
        assert x[f].dtype == y[f].dtype, (ctx, f, x[f].dtype, y[f].dtype)
        assert np.array_equal(x[f], y[f]), (ctx, f)


def as_out(e):
    return {"ids": e.ids, "off": e.off, "pos_start": e.pos_start, "pos_end": e.pos_end, "changed": e.changed,
            "branch_rewritten": e.branch_rewritten}


def expected(g, genes={}):
    """correct_loop's answer for graph g: the lazy graph's device arrays, or a host-edited graph's objects"""
    src = g._source_encoded()
    if g._on_device():
        a = g._require_device_state().arrays()
        w = a
        ranks = g._gene_ranks(list(genes))
        amr = np.isin(np.abs(a["node_key"]), ranks).any(axis=1) if ranks and len(a["node_key"]) else \
            np.zeros(len(a["node_cov"]), bool)
    else:
        a, w = g._unitig_index_arrays(), g._read_index_arrays()
        rank = {n: i + 1 for i, n in enumerate(g._vocab.names)}
        w["node_key"] = np.asarray([[x.get_strand() * rank[x.get_name()] for x in n.get_canonical_geneMer()]
                                    for n in g._nodes.values()], np.int64).reshape(len(g._nodes), -1)
        amr_nodes = g.get_AMR_nodes(genes)
        amr = np.asarray([nh in amr_nodes for nh in g._nodes], bool)
    u = unitig_loop(a)
    bub = bubble_loop(a, u, read_path_loop({**a, **w}, u))
    return correct_loop({**a, **w}, u, bub, src.ids, src.off, src.pos_start, src.pos_end, replace_loop(u, bub, amr))


def corrected(reads, k, genes={}, positions=None):
    """correct_compacted_bubbles on a lazy graph, checked against correct_loop"""
    g = construct_graph.GeneMerGraph(reads, k, positions)
    e = g.correct_compacted_bubbles(genes)
    same(as_out(e), expected(g, genes))
    assert g.__dict__["_lazy"]
    return e


def graph_summary(g):
    return ({h: n.get_node_coverage() for h, n in g.get_nodes().items()},
            {h: e.get_edge_coverage() for h, e in g.get_edges().items()})


@pytest.mark.parametrize("err", [ERR_SUB, ERR_DEL, ERR_INS])
def test_one_error_is_corrected_and_the_rebuild_is_the_true_graph(fake_device, err):
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": err}
    e = corrected(reads, 3)
    assert e.reads["e"] == TRUE and e.changed.tolist() == [0] * 5 + [1]
    assert e.branch_rewritten.tolist() == [0, 1]
    g = construct_graph.GeneMerGraph(e, 3)
    truth = construct_graph.GeneMerGraph({**{"t%d" % i: TRUE for i in range(6)}}, 3)
    assert graph_summary(g) == graph_summary(truth)
    assert g.compacted_bubbles()["branch_off"].tolist() == [0]


def test_strand_flip_and_a_read_that_crosses_backwards(fake_device):
    flip = ["+a", "+b", "+c", "-d", "+e", "+f", "+g"]
    e = corrected({**{"t%d" % i: TRUE for i in range(5)}, "e": flip}, 3)
    assert e.reads["e"] == TRUE
    e = corrected({**{"t%d" % i: TRUE for i in range(3)}, **{"r%d" % i: rc(TRUE) for i in range(2)}, "e": rc(ERR_SUB),
                   "f": ERR_DEL}, 3)
    assert e.reads["e"] == rc(TRUE) and e.reads["f"] == TRUE


def test_two_bubbles_of_one_read_share_a_junction(fake_device):
    true = ["+%s" % c for c in "abcdefghijk"]
    err = list(true)
    err[3], err[7] = "+x", "+y"                                # the sink window of one is the source of the other
    e = corrected({**{"t%d" % i: true for i in range(5)}, "e": err}, 3)
    assert e.reads["e"] == true and sorted(e.branch_rewritten.tolist()) == [0, 0, 1, 1]


def test_three_branches(fake_device):
    e = corrected({**{"t%d" % i: TRUE for i in range(5)}, "e1": ERR_SUB, "e2": ["+a", "+b", "+c", "+y", "+e", "+f", "+g"]}, 3)
    assert e.reads["e1"] == TRUE and e.reads["e2"] == TRUE and e.branch_rewritten.tolist() == [0, 1, 1]


def test_a_read_that_starts_on_the_branch_is_counted_not_rewritten(fake_device):
    start = ERR_SUB[1:]
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": ERR_SUB, "s": start}
    g = construct_graph.GeneMerGraph(reads, 3)
    assert g.compacted_bubbles()["branch_reads"].tolist() == [5, 2]
    e = corrected(reads, 3)
    assert e.reads["s"] is reads["s"] and e.reads["e"] == TRUE and e.branch_rewritten.tolist() == [0, 1]


def test_an_edge_filtered_away_next_to_a_branch(fake_device):
    """q enters the error branch from z; filter_graph(1, 2) deletes z -> branch (coverage 1) but keeps z's window: a
    live neighbour window that is not the bubble's source, so q is not rewritten"""
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e1": ERR_SUB, "e2": ERR_SUB, "q": ["+z"] + ERR_SUB[1:]}
    g = construct_graph.GeneMerGraph(reads, 3)
    g.filter_graph(1, 2)
    e = g.correct_compacted_bubbles()
    same(as_out(e), expected(g))
    assert e.branch_rewritten.tolist() == [0, 2] and e.changed.tolist() == [0] * 5 + [1, 1, 0]


def test_a_branch_with_a_gene_of_interest_is_spared(fake_device):
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": ERR_SUB}
    e = corrected(reads, 3, {"x"})
    assert not e.changed.any() and e.reads == reads
    assert corrected(reads, 3, {"q"}).reads["e"] == TRUE


def test_a_circle(fake_device):
    loop = ["+a", "+b", "+c", "+d", "+e", "+f", "+g", "+a", "+b", "+c"]
    err = list(loop)
    err[4] = "+x"
    e = corrected({**{"t%d" % i: loop for i in range(4)}, "e": err}, 3)
    assert e.reads["e"] == loop


def test_positions_policy(fake_device):
    pos = lambda read: [(10 * i, 10 * i + 5) for i in range(len(read))]
    for err, want in ((ERR_DEL, [(0, 5), (10, 15), (20, 25), (20, 25), (30, 35), (40, 45), (50, 55)]),
                      (ERR_INS, [(0, 5), (10, 15), (20, 25), (40, 45), (50, 55), (60, 65), (70, 75)])):
        # deletion: calls 1, 2 (b, c) become b, c, d, and the extra call takes the positions of the last replaced
        # call; insertion: calls 1..3 (b, c, x) become b, c, and new call j takes those of replaced call j
        reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": err}
        positions = {r: pos(x) for r, x in reads.items()}
        e = corrected(reads, 3, positions=positions)
        assert e.reads["e"] == TRUE and e.positions["e"] == want
        assert e.positions["t0"] is positions["t0"]


def test_the_source_reads_are_left_untouched_and_save_load(fake_device, tmp_path):
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": ERR_SUB, "f": rc(ERR_SUB)}
    src = encode.EncodedReads(reads)
    before = copy.deepcopy((src.reads, src.ids, src.off, src.read_ids, src.vocab.names))
    g = construct_graph.GeneMerGraph(src, 3)
    e = g.correct_compacted_bubbles()
    after = (src.reads, src.ids, src.off, src.read_ids, src.vocab.names)
    assert all(np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y for x, y in zip(before, after))
    assert g._encoded is src and e.vocab is src.vocab and e.read_ids is src.read_ids and e.reads is not src.reads
    assert e.reads["e"] == TRUE and e.reads["f"] == rc(TRUE) and e.reads["t0"] is reads["t0"]
    e.save(str(tmp_path / "c.npz"))
    back = encode.EncodedReads.load(str(tmp_path / "c.npz"))
    assert back.reads == e.reads and np.array_equal(back.ids, e.ids) and np.array_equal(back.off, e.off)


def test_loop_device_path(loop_device):
    """the lazy path through the double's correct_bubble_reads gives the same as the host implementation"""
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": ERR_SUB, "f": rc(ERR_DEL)}
    e = corrected(reads, 3)
    assert e.reads["e"] == TRUE and e.reads["f"] == rc(TRUE)


def test_host_implementation_against_the_loop(fake_device):
    """random graphs of reads with errors, lazy and host-edited, before and after filter_graph,
    remove_short_linear_paths and remove_node; with and without a gene of interest"""
    n = n_changed = 0
    for seed in range(300):
        rng = np.random.default_rng(47000 + seed)
        reads = error_reads(rng)
        k = int(rng.integers(1, 4))
        genes = {"x0"} if seed % 4 == 0 else {}
        try:
            lazy = construct_graph.GeneMerGraph(reads, k)
            hst = construct_graph.GeneMerGraph(reads, k)
            ops = [[], [("filter_graph", (2, 1))], [("filter_graph", (1, 2))], [("remove_short_linear_paths", (3,))]][seed % 4]
            for g in (lazy, hst):
                for op, args in ops:
                    getattr(g, op)(*args)
            hst._touch()
            if seed % 5 == 1 and len(hst.get_nodes()):
                objs = list(hst.get_nodes().values())
                hst.remove_node(objs[int(rng.integers(len(objs)))])
            x = lazy.correct_compacted_bubbles(genes)
            y = hst.correct_compacted_bubbles(genes)
        except (AssertionError, TypeError):                    # palindromic window, a removal that meets a multi-edge
            continue
        same(as_out(x), expected(lazy, genes), seed)
        same(as_out(y), expected(hst, genes), (seed, "host"))
        n_changed += int(x.changed.any())
        n += 1
    assert n >= 200 and n_changed >= 30, (n, n_changed)


@pytest.mark.parametrize("name", FIXTURES)
def test_host_implementation_on_fixtures(fake_device, name):
    from tests.helpers import load_input, read_dict
    vocab, ids, off, ps, pe = load_input(name)
    reads, pos = read_dict(vocab, ids, off, ps, pe)
    for k in (1, 3, 5):
        try:
            g = construct_graph.GeneMerGraph(reads, k, pos)
        except AssertionError:
            continue
        same(as_out(g.correct_compacted_bubbles()), expected(g), (name, k))


def test_empty_graph(fake_device):
    g = construct_graph.GeneMerGraph({}, 3)
    e = g.correct_compacted_bubbles()
    assert e.reads == {} and e.off.tolist() == [0] and len(e.ids) == 0


def test_bad_replace_with_raises():
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": ERR_SUB}
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    dev = CorrectionDevice().build(ids, off, 3)
    a = dev.arrays()
    u = unitig_loop(a)
    bub = bubble_loop(a, u, read_path_loop(a, u))
    src = encode.EncodedReads(reads)
    for rw in ([-1, 1], [2, -1], [-2, 0], [-1]):
        with pytest.raises(ValueError):
            dev.correct_bubble_reads(np.asarray(rw))
        if len(rw) == 2:
            with pytest.raises(ValueError):
                construct_graph.GeneMerGraph._corrected_reads_over(u, read_path_loop(a, u), bub, a, a["node_key"],
                                                                   np.asarray(rw), src)


UPSTREAM = os.environ.get("AMIRA_REFERENCE_ROOT", "/root/reference")


@pytest.mark.skipif(not os.path.isfile(os.path.join(UPSTREAM, "amira", "construct_graph.py")),
                    reason="upstream checkout not present")
def test_correction_methods_are_not_upstream_names():
    """bind_upstream overrides upstream's methods by name: the new methods must not replace one of upstream's"""
    import ast
    with open(os.path.join(UPSTREAM, "amira", "construct_graph.py")) as f:
        tree = ast.parse(f.read())
    cls = [c for c in tree.body if isinstance(c, ast.ClassDef) and c.name == "GeneMerGraph"]
    assert len(cls) == 1
    names = {f.name for f in cls[0].body if isinstance(f, (ast.FunctionDef, ast.AsyncFunctionDef))}
    assert names and not names & {"correct_compacted_bubbles", "_corrected_reads_over", "_source_encoded",
                                  "_bubble_winners"}
