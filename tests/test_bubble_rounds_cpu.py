"""correct_bubbles_until_stable without a GPU: the orchestration over the test double with the device policy
(PolicyDevice, tests/bubble_rounds_reference.py) against rounds_loop, its definition as a composition of existing
methods, round by round: the per round counts, the reads, the CSR, the changed union and the final graph.  Random
error and random reads that need two rounds or more, the smallest of them pinned by hand; max_rounds 0 and 1, a graph
without bubbles, an empty read set, spared genes, positions carried through, filter_graph, a host-edited graph against
the lazy one, and the source graph left as it was."""
import numpy as np
import pytest

from amira_b200 import construct_graph, encode
from oracle import gmg_oracle as O
from tests.bubble_rounds_reference import PolicyDevice, rounds_loop
from tests.test_bubbles_cpu import TRUE, error_reads
from tests.test_random_small_cpu import random_reads

FIELDS = ("ids", "off", "pos_start", "pos_end")


@pytest.fixture
def policy_device(monkeypatch):
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", PolicyDevice)


def state(g):
    """what correct_bubbles_until_stable must leave as it was"""
    arrays = g._require_device_state().arrays() if g._on_device() else \
        ({h: n.get_node_coverage() for h, n in g._nodes.items()}, {h: e.get_edge_coverage() for h, e in g._edges.items()})
    return g._device_ops, g._encoded, dict(g._reads), g._minNodeCoverage, g._minEdgeCoverage, arrays


def same_state(x, y):
    assert x[:5] == y[:5]
    if isinstance(x[5], dict):
        assert O.diff_arrays(x[5], y[5]) == []
    else:
        assert x[5] == y[5]


def until_stable(g, max_rounds=30, genes={}, filt=None):
    """the product against rounds_loop; returns (graph, reads)"""
    before = state(g)
    graph, reads = g.correct_bubbles_until_stable(max_rounds, genes, filt)
    assert graph is g or graph.__dict__["_lazy"]
    same_state(state(g), before)
    want_g, want_e, want_changed, want_rounds = rounds_loop(g, max_rounds, genes, filt)
    assert reads.rounds == want_rounds
    assert reads.reads == want_e.reads and reads.positions == want_e.positions
    for f in FIELDS:
        x, y = getattr(reads, f), getattr(want_e, f)
        assert (x is None and y is None) or np.array_equal(x, y), f
    assert np.array_equal(reads.changed, want_changed)
    assert reads.vocab.names == g._source_encoded().vocab.names and reads.read_ids == list(g._reads)
    if want_g is g:
        assert graph is g
    else:
        assert graph is not g and graph._device_ops == want_g._device_ops
        assert (graph._minNodeCoverage, graph._minEdgeCoverage) == (want_g._minNodeCoverage, want_g._minEdgeCoverage)
        assert O.diff_arrays(graph._arrays(), want_g._arrays()) == []       # graph rebuilds itself: the replayed filter
        assert np.array_equal(reads.branch_rewritten, want_e.branch_rewritten)
    return graph, reads


def rc(read):
    return [("-" if g[0] == "+" else "+") + g[1:] for g in read[::-1]]


# a substitution (e1) inside the stretch that a longer detour (e2) replaces: the detour's bubble exists only once the
# substitution is corrected, so round 1 corrects e1 and round 2 corrects e2
T = ["+%s" % c for c in ("s0", "s1", "a", "b", "c", "d", "e", "f", "g", "h", "i", "j", "t0", "t1")]
TWO_ROUNDS = {**{"t%d" % i: T for i in range(5)}, "e1": T[:7] + ["+x"] + T[8:], "e2": T[:4] + ["+p", "+q", "+r", "+u", "+v", "+w"] + T[10:]}
TWO_ROUNDS_K = 3
# the smallest input (by call count) that needs two rounds among nested_reads(np.random.default_rng(s)) for s in
# 53000..53199, each at the k the same generator draws next: s = 53008, k = 1
SMALLEST = {"t0": ["+g6", "+g0", "-g2", "+g5", "-g1", "-g7", "-g4", "-g3"],
            "t1": ["+g3", "+g4", "+g7", "+g1", "-g5", "+g2", "-g0", "-g6"],
            "t2": ["+g3", "+g4", "+g7", "+g1", "-g5", "+g2", "-g0", "-g6"],
            "e1": ["+g3", "+g4", "+g7", "+x0", "-g5", "+g2", "-g0", "-g6"],
            "e2": ["+g3", "+y0", "+y1", "+y2", "-g5", "+g2", "-g0", "-g6"]}


def nested_reads(rng):
    """copies of a random gene sequence (some reverse complemented), one read with a substitution and one with a
    detour around it"""
    n = int(rng.integers(8, 16))
    truth = [("+" if rng.random() < 0.5 else "-") + "g%d" % i for i in rng.permutation(n)]
    reads = {"t%d" % r: (rc(truth) if rng.random() < 0.3 else list(truth)) for r in range(int(rng.integers(3, 6)))}
    i = int(rng.integers(3, n - 3))
    inner = list(truth)
    inner[i] = "+x0"
    lo, hi = int(rng.integers(1, i)), int(rng.integers(i + 1, n - 1))
    reads["e1"] = rc(inner) if rng.random() < 0.3 else inner
    reads["e2"] = truth[:lo] + ["+y%d" % j for j in range(int(rng.integers(1, 6)))] + truth[hi:]
    return reads


def edit_rounds(reads):
    return sum(r["steps"] > 0 for r in reads.rounds)


def test_two_rounds(policy_device):
    graph, reads = until_stable(construct_graph.GeneMerGraph(TWO_ROUNDS, TWO_ROUNDS_K))
    assert [r["steps"] for r in reads.rounds] == [1, 1, 0] and reads.rounds[-1]["bubbles"] == 0
    assert reads.reads["e1"] == T and reads.reads["e2"] == T and reads.changed.tolist() == [0] * 5 + [1, 1]
    assert graph.compacted_bubbles()["branch_off"].tolist() == [0]
    rng = np.random.default_rng(53008)
    assert nested_reads(rng) == SMALLEST and int(rng.integers(1, 5)) == 1
    graph, reads = until_stable(construct_graph.GeneMerGraph(SMALLEST, 1))
    assert edit_rounds(reads) == 2


def test_sweep_needs_two_rounds_or_more(policy_device):
    """nested errors, error reads and random reads, some after filter_graph(1, 2)"""
    n = multi = 0
    for seed in range(150):
        rng = np.random.default_rng(53000 + seed)
        reads = [nested_reads, error_reads,
                 lambda r: random_reads(r, int(r.integers(1, 25)), int(r.integers(2, 9)), int(r.integers(1, 14)))][seed % 3](rng)
        k = int(rng.integers(1, 5))
        try:
            g = construct_graph.GeneMerGraph(reads, k)
        except AssertionError:                                 # palindromic window
            continue
        graph, out = until_stable(g, filt=(1, 2) if seed % 7 == 0 else None)
        n += 1
        multi += edit_rounds(out) >= 2
    assert n >= 100 and multi >= 8, (n, multi)


def test_max_rounds_zero_and_one(policy_device):
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": ["+a", "+b", "+c", "+x", "+e", "+f", "+g"]}
    g = construct_graph.GeneMerGraph(reads, 3)
    graph, out = until_stable(g, max_rounds=0)
    assert graph is g and out.rounds == [] and not out.changed.any() and out.reads == reads
    assert out.reads is not g._reads
    graph, out = until_stable(g, max_rounds=1)
    assert graph is not g and len(out.rounds) == 1 and out.reads["e"] == TRUE and out.changed.tolist() == [0] * 5 + [1]
    graph, out = until_stable(construct_graph.GeneMerGraph(TWO_ROUNDS, TWO_ROUNDS_K), max_rounds=1)
    assert len(out.rounds) == 1 and out.reads["e1"] == T and out.reads["e2"] == TWO_ROUNDS["e2"]
    assert graph.compacted_bubbles()["branch_off"].tolist() == [0, 2]


def test_without_bubbles_the_graph_is_self(policy_device):
    g = construct_graph.GeneMerGraph({"r%d" % i: TRUE for i in range(4)}, 3)
    graph, out = until_stable(g)
    assert graph is g and out.rounds == [{"bubbles": 0, "branches": 0, "replaced": 0, "steps": 0, "reads": 0, "calls": 28}]
    assert out.branch_rewritten.tolist() == [] and out.reads == g._reads


def test_empty_read_set(policy_device):
    g = construct_graph.GeneMerGraph({}, 3)
    graph, out = g.correct_bubbles_until_stable()
    assert graph is g and out.reads == {} and out.off.tolist() == [0] and len(out.ids) == 0
    assert out.rounds == [{"bubbles": 0, "branches": 0, "replaced": 0, "steps": 0, "reads": 0, "calls": 0}]


def test_spared_genes(policy_device):
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": ["+a", "+b", "+c", "+x", "+e", "+f", "+g"]}
    g = construct_graph.GeneMerGraph(reads, 3)
    graph, out = until_stable(g, genes={"x"})
    assert graph is g and out.rounds[0]["replaced"] == 0 and out.reads == reads
    graph, out = until_stable(construct_graph.GeneMerGraph(TWO_ROUNDS, TWO_ROUNDS_K), genes={"x"})
    assert out.reads["e1"] == TWO_ROUNDS["e1"] and [r["steps"] for r in out.rounds] == [0]


def test_positions_are_carried_through(policy_device):
    positions = {r: [(10 * i, 10 * i + 5) for i in range(len(x))] for r, x in TWO_ROUNDS.items()}
    g = construct_graph.GeneMerGraph(TWO_ROUNDS, TWO_ROUNDS_K, positions)
    graph, out = until_stable(g)
    assert out.positions["t0"] is positions["t0"] and out.positions["e1"] == positions["e1"]
    assert len(out.positions["e2"]) == len(T) and set(out.positions["e2"]) <= set(positions["e2"])
    assert out.positions["e2"] == sorted(out.positions["e2"]) and np.array_equal(out.pos_start[out.off[-2]:], [p for p, _ in out.positions["e2"]])
    assert graph._genePositions is out.positions


def test_filter_graph(policy_device):
    for filt in ((3, 1), (1, 2), (2, 2), (10**6, 1)):
        g = construct_graph.GeneMerGraph(TWO_ROUNDS, TWO_ROUNDS_K)
        graph, out = until_stable(g, filt=filt)
        assert graph is not g and (graph._minNodeCoverage, graph._minEdgeCoverage) == filt
        assert graph._device_ops == (("filter_graph", filt),)


def test_host_edited_against_lazy(policy_device):
    """round 1 on the host implementation of a host-edited graph, then rounds on the handle, against the reference and
    against the same loop from the lazy graph"""
    n = edited = 0
    for seed in range(40):
        rng = np.random.default_rng(52000 + seed)
        reads = nested_reads(rng) if seed % 3 else error_reads(rng)
        k = int(rng.integers(1, 4))
        genes = {"g1"} if seed % 3 == 0 else {}
        try:
            lazy, hst = construct_graph.GeneMerGraph(reads, k), construct_graph.GeneMerGraph(reads, k)
        except AssertionError:                                 # palindromic window
            continue
        for g in (lazy, hst):
            g.filter_graph(1, 2 if seed % 4 == 0 else 1)
        hst._touch()
        a = until_stable(lazy, genes=genes)
        b = until_stable(hst, genes=genes)
        assert a[1].rounds == b[1].rounds and a[1].reads == b[1].reads, seed
        assert np.array_equal(a[1].ids, b[1].ids) and np.array_equal(a[1].off, b[1].off), seed
        assert np.array_equal(a[1].changed, b[1].changed), seed
        n += 1
        edited += edit_rounds(b[1]) >= 1
    assert n >= 30 and edited >= 10, (n, edited)


def test_encoded_source_is_left_as_it_was(policy_device):
    src = encode.EncodedReads(dict(TWO_ROUNDS))
    ids, off = src.ids.copy(), src.off.copy()
    g = construct_graph.GeneMerGraph(src, TWO_ROUNDS_K)
    graph, out = until_stable(g)
    assert g._encoded is src and np.array_equal(src.ids, ids) and np.array_equal(src.off, off)
    assert not hasattr(src, "rounds") and src.reads == TWO_ROUNDS and graph._encoded is out
