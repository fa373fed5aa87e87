"""Simple bubbles without a GPU: the invariants of bubble_loop (tests/bubble_reference.py, the reference of the GPU
tests) on random tiny graphs, graphs of reads with gene-call errors, the fixtures and hand-made probes with known
answers (a substitution, a deletion and a strand flip at k = 3, three branches, one source end with two bubbles, a
bubble read in both orientations, source and sink on one unitig, a turn-back, a self edge, overlapping errors, a
circle); the product's host implementation (GeneMerGraph._bubbles_over) against the loop on lazy graphs through the
test double and on host-edited graphs, after filters, trimming and remove_node; pop_compacted_bubbles against
pop_loop, on the device-style path and the host path."""
import os

import numpy as np
import pytest

from amira_b200 import construct_graph
from oracle import gmg_oracle as O
from tests.bubble_reference import BubbleDevice, bubble_loop, pop_loop
from tests.fake_device import OracleBackedDevice
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES, same
from tests.unitig_path_reference import read_path_loop
from tests.unitig_reference import unitig_loop

TRUE = ["+a", "+b", "+c", "+d", "+e", "+f", "+g"]


@pytest.fixture
def fake_device(monkeypatch):
    """lazy graphs on the test double without the new call: served by the host implementation over its arrays"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", OracleBackedDevice)


def host():
    return construct_graph.GeneMerGraph.__new__(construct_graph.GeneMerGraph)


def error_reads(rng, n_reads=None):
    """reads along one or two random gene sequences, with substitutions, deletions and strand flips: the structures
    bubbles come from"""
    genes = ["g%d" % i for i in range(int(rng.integers(8, 20)))]
    seqs = [[("+" if rng.random() < 0.5 else "-") + g for g in rng.permutation(genes)[:int(rng.integers(6, len(genes) + 1))]]
            for _ in range(int(rng.integers(1, 3)))]
    reads = {}
    for r in range(n_reads or int(rng.integers(6, 24))):
        s = seqs[int(rng.integers(len(seqs)))]
        lo = int(rng.integers(0, 3))
        read = list(s[lo:len(s) - int(rng.integers(0, 3))])
        if rng.random() < 0.5:
            read = [("-" if g[0] == "+" else "+") + g[1:] for g in read[::-1]]
        for _ in range(int(rng.integers(0, 2))):
            i, kind = int(rng.integers(len(read))), rng.random()
            if kind < 0.4:
                read[i] = "+x%d" % int(rng.integers(3))
            elif kind < 0.7 and len(read) > 2:
                del read[i]
            else:
                read[i] = ("-" if read[i][0] == "+" else "+") + read[i][1:]
        reads["r%d" % r] = read
    return reads


def check_bubbles(a, u, p, bub):
    """two branches or more per bubble, sigma < tau ^ 1, no unitig twice, every branch a walk from sigma through its
    whole unitig to tau, and branch_reads the full-length steps on it"""
    off = bub["branch_off"]
    B = len(bub["source"])
    assert len(bub["sink"]) == B and len(off) == B + 1 and off[0] == 0 and off[-1] == len(bub["branch_unitig"])
    assert (np.diff(off) >= 2).all()
    assert (bub["source"] < (bub["sink"] ^ 1)).all()
    assert len(set(bub["branch_unitig"].tolist())) == len(bub["branch_unitig"])
    assert (np.diff(bub["source"]) >= 0).all()
    fw_off, fw_edges, bw_off, bw_edges = (a[f].tolist() for f in ("fw_off", "fw_edges", "bw_off", "bw_edges"))
    tgt, td = a["edge_tgt"].tolist(), a["edge_td"].tolist()
    uoff, unodes = u["unitig_off"].tolist(), u["unitig_nodes"].tolist()

    def lst(s):
        n = s >> 1
        return fw_edges[fw_off[n]:fw_off[n + 1]] if s & 1 == 0 else bw_edges[bw_off[n]:bw_off[n + 1]]

    def step(s, n):
        """the edge of list(s) into node n, and the state it continues through"""
        e = [j for j in lst(s) if tgt[j] == n]
        assert len(e) >= 1
        return 2 * n + (1 if td[e[0]] < 0 else 0)

    ulen = np.diff(u["unitig_off"])
    full = np.bincount(p["unitig"][p["length"] == ulen[p["unitig"]]], minlength=len(ulen))
    for i in range(B):
        sigma, tau = int(bub["source"][i]), int(bub["sink"][i])
        for g in range(off[i], off[i + 1]):
            b, o = int(bub["branch_unitig"][g]), int(bub["branch_orient"][g])
            nodes = unodes[uoff[b]:uoff[b + 1]]
            if o == -1:
                nodes = nodes[::-1]
            assert not u["circular"][b] and (sigma >> 1) not in nodes and (tau >> 1) not in nodes
            s = sigma
            for n in nodes:
                s = step(s, n)
            assert step(s, tau >> 1) == tau, (i, g)
            assert bub["branch_reads"][g] == full[b]


def checked(a):
    u = unitig_loop(a)
    p = read_path_loop(a, u)
    bub = bubble_loop(a, u, p)
    check_bubbles(a, u, p, bub)
    same(host()._bubbles_over(a, a), bub)
    return u, bub


def build(reads, k):
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    return BubbleDevice().build(ids, off, k)


@pytest.mark.parametrize("k", [1, 2, 3])
def test_bubble_invariants_on_random_tiny_graphs(k):
    n = n_bub = 0
    for seed in range(3000):
        if n == 200:
            break
        rng = np.random.default_rng(41000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14))) \
            if seed % 2 else error_reads(rng)
        try:
            dev = build(reads, k)
        except AssertionError:                                 # palindromic window
            continue
        _, bub = checked(dev.arrays())
        n_bub += len(bub["source"])
        flags = (rng.random(dev.sizes()["nodes"]) < 0.2).astype(np.uint8)
        try:
            dev.remove_nodes(flags)
        except TypeError:                                      # a removal meets a multi-edge
            continue
        checked(dev.arrays())
        n += 1
    assert n == 200 and n_bub >= 20, n_bub


@pytest.mark.parametrize("name", FIXTURES)
def test_bubble_invariants_on_fixtures(name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    for k in (1, 3, 5):
        try:
            dev = BubbleDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        checked(dev.arrays())


def one_bubble(reads, k):
    a = build(reads, k).arrays()
    u, bub = checked(a)
    return a, u, bub


@pytest.mark.parametrize("err,lengths", [(["+a", "+b", "+c", "+x", "+e", "+f", "+g"], [3, 3]),
                                         (["+a", "+b", "+c", "+e", "+f", "+g"], [3, 2]),
                                         (["+a", "+b", "+c", "-d", "+e", "+f", "+g"], [3, 3])])
def test_one_error_makes_one_bubble(err, lengths):
    """five correct reads and one with a substitution, a deletion or a strand flip: one bubble, the true branch first
    in its list here, with coverages 15 against the error's, and the reads that run each branch"""
    a, u, bub = one_bubble({**{"t%d" % i: TRUE for i in range(5)}, "e": err}, 3)
    assert len(bub["source"]) == 1 and bub["branch_off"].tolist() == [0, 2]
    bu = bub["branch_unitig"]
    assert np.diff(u["unitig_off"])[bu].tolist() == lengths
    assert u["cov_sum"][bu].tolist() == [15, lengths[1]]
    assert bub["branch_reads"].tolist() == [5, 1]


def test_three_branches():
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e1": ["+a", "+b", "+c", "+x", "+e", "+f", "+g"],
             "e2": ["+a", "+b", "+c", "+y", "+e", "+f", "+g"]}
    _, u, bub = one_bubble(reads, 3)
    assert bub["branch_off"].tolist() == [0, 3] and bub["branch_reads"].tolist() == [5, 1, 1]


def test_one_source_end_two_bubbles():
    """a junction whose list holds branches to two different sinks: two bubbles from one source, in the list order of
    their first branch"""
    reads = {"r1": ["+s", "+x1", "+t"], "r2": ["+s", "+y1", "+w"], "r3": ["+s", "+x2", "+t"], "r4": ["+s", "+y2", "+w"]}
    a, u, bub = one_bubble(reads, 1)
    assert len(bub["source"]) == 2 and bub["source"][0] == bub["source"][1] and bub["sink"][0] != bub["sink"][1]
    assert bub["branch_off"].tolist() == [0, 2, 4]
    first = u["unitig_nodes"][u["unitig_off"][bub["branch_unitig"]]].tolist()     # one-node branches
    assert first == [1, 5, 3, 6]                                                 # x1, x2 | y1, y2 by first seen


def test_bubble_read_both_ways_is_reported_once():
    fw = {"t%d" % i: TRUE for i in range(3)}
    rev = {"r%d" % i: [("-" if g[0] == "+" else "+") + g[1:] for g in TRUE[::-1]] for i in range(2)}
    err = ["+a", "+b", "+c", "+x", "+e", "+f", "+g"]
    _, u, bub = one_bubble({**fw, **rev, "e": [("-" if g[0] == "+" else "+") + g[1:] for g in err[::-1]]}, 3)
    assert len(bub["source"]) == 1 and bub["branch_reads"].tolist() == [5, 1]


def test_source_and_sink_on_one_unitig():
    """the path leaves a unitig and comes back into the same unitig: x and y on one unitig, other than the branches"""
    reads = {"t1": ["+a", "+b", "+c", "+a", "+b"], "t2": ["+a", "+b", "+x", "+a", "+b"]}
    a, u, bub = one_bubble(reads, 1)
    assert len(bub["source"]) == 1
    assert u["node_unitig"][bub["source"][0] >> 1] == u["node_unitig"][bub["sink"][0] >> 1]


def test_no_bubble_cases():
    """a turn-back (two branches from one end back into it), a one-node branch with a self edge, two overlapping
    errors on different reads (the branches are not single unitigs), and a circle"""
    for reads, k in (({"t1": ["+a", "+b", "+c"], "t2": ["+a", "+b", "-b", "-a"], "t3": ["+a", "+b", "+d", "-b", "-a"]}, 1),
                     ({"t1": ["+a", "+b", "+b", "+c"], "t2": ["+a", "+x", "+c"]}, 1),
                     ({**{"t%d" % i: TRUE for i in range(4)}, "e1": ["+a", "+b", "+c", "+x", "+e", "+f", "+g"],
                       "e2": ["+a", "+b", "+c", "+d", "+y", "+f", "+g"]}, 3),
                     ({"r1": ["+a", "+b", "+c"] * 3 + ["+a"]}, 1)):
        _, _, bub = one_bubble(reads, k)
        assert len(bub["source"]) == 0, reads


def test_empty_graph_has_no_bubbles(fake_device):
    g = construct_graph.GeneMerGraph({}, 3)
    bub = g.compacted_bubbles()
    assert bub["branch_off"].tolist() == [0] and all(len(bub[f]) == 0 for f in bub if f != "branch_off")
    assert g.pop_compacted_bubbles() == []


def node_keys(g):
    return sorted(tuple(g_.get_name() for g_ in n.get_canonical_geneMer()) for n in g.get_nodes().values())


def test_pop_substitution_gives_the_true_graph(fake_device):
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": ["+a", "+b", "+c", "+x", "+e", "+f", "+g"]}
    for lazy in (True, False):
        g = construct_graph.GeneMerGraph(reads, 3)
        if not lazy:
            g._touch()
        removed = g.pop_compacted_bubbles()
        assert len(removed) == 3 and (g.__dict__["_lazy"] or not lazy)
        assert len(g.compacted_unitigs()["circular"]) == 1
        assert g.compacted_bubbles()["branch_off"].tolist() == [0]
        assert node_keys(g) == node_keys(construct_graph.GeneMerGraph({r: reads[r] for r in reads if r != "e"}, 3))
        assert g.get_reads_to_correct() == {"e"}


def test_pop_keeps_a_branch_with_a_gene_of_interest(fake_device):
    reads = {**{"t%d" % i: TRUE for i in range(5)}, "e": ["+a", "+b", "+c", "+x", "+e", "+f", "+g"]}
    for lazy in (True, False):
        g = construct_graph.GeneMerGraph(reads, 3)
        if not lazy:
            g._touch()
        assert g.pop_compacted_bubbles({"x"}) == []
        assert len(g.compacted_bubbles()["source"]) == 1


def test_pop_lazy_and_host_paths_agree(fake_device):
    """random graphs with errors, lazy (the policy over the double's arrays, removal on the double) against
    host-edited (the same policy over the objects, remove_node): the same hashes in the same order, the loop's
    answer, and the same graph afterwards; also after filter_graph and remove_short_linear_paths"""
    n = n_popped = 0
    for seed in range(300):
        rng = np.random.default_rng(43000 + seed)
        reads = error_reads(rng)
        k = int(rng.integers(1, 4))
        genes = {"x0"} if seed % 3 == 0 else {}
        try:
            lazy = construct_graph.GeneMerGraph(reads, k)
        except AssertionError:
            continue
        ops = [[], [("filter_graph", (2, 1))], [("remove_short_linear_paths", (3,))]][seed % 3]
        hst = construct_graph.GeneMerGraph(reads, k)
        try:
            for g in (lazy, hst):
                for op, args in ops:
                    getattr(g, op)(*args)
            hst._touch()
            a = lazy._require_device_state().arrays()
            u = unitig_loop(a)
            bub = bubble_loop(a, u, read_path_loop(a, u))
            same(lazy.compacted_bubbles(), bub, seed)
            same(hst.compacted_bubbles(), bub, (seed, "host"))
            ranks = lazy._gene_ranks(list(genes))
            amr = lazy._require_device_state().nodes_containing(ranks) if ranks else np.zeros(len(u["node_unitig"]), bool)
            want = pop_loop(u, bub, np.asarray(amr, bool))
            got_lazy = lazy.pop_compacted_bubbles(genes)
            got_host = hst.pop_compacted_bubbles(genes)
        except TypeError:                                      # a removal meets a multi-edge, as upstream's does
            continue
        assert lazy.__dict__["_lazy"] or not len(want)
        assert got_lazy == got_host, seed
        assert len(got_lazy) == len(want)
        assert sorted(lazy.get_nodes()) == sorted(hst.get_nodes()), seed
        assert lazy.get_reads_to_correct() == hst.get_reads_to_correct(), seed
        n_popped += bool(want)
        n += 1
    assert n >= 200 and n_popped >= 20, (n, n_popped)


def test_bubbles_after_host_remove_node(fake_device):
    n = 0
    for seed in range(100):
        rng = np.random.default_rng(44000 + seed)
        reads = error_reads(rng)
        try:
            g = construct_graph.GeneMerGraph(reads, 2)
        except AssertionError:
            continue
        objs = list(g.get_nodes().values())
        try:
            for i in rng.choice(len(objs), min(len(objs), 2), replace=False).tolist():
                g.remove_node(objs[i])
        except TypeError:
            continue
        a = g._unitig_index_arrays()
        a.update(g._read_index_arrays())
        u = unitig_loop(a)
        p = read_path_loop(a, u)
        bub = bubble_loop(a, u, p)
        check_bubbles(a, u, p, bub)
        same(g.compacted_bubbles(), bub, seed)
        n += 1
    assert n >= 50


UPSTREAM = os.environ.get("AMIRA_REFERENCE_ROOT", "/root/reference")


@pytest.mark.skipif(not os.path.isfile(os.path.join(UPSTREAM, "amira", "construct_graph.py")),
                    reason="upstream checkout not present")
def test_bubble_methods_are_not_upstream_names():
    """bind_upstream overrides upstream's methods by name: the new methods must not replace one of upstream's"""
    import ast
    with open(os.path.join(UPSTREAM, "amira", "construct_graph.py")) as f:
        tree = ast.parse(f.read())
    cls = [c for c in tree.body if isinstance(c, ast.ClassDef) and c.name == "GeneMerGraph"]
    assert len(cls) == 1
    names = {f.name for f in cls[0].body if isinstance(f, (ast.FunctionDef, ast.AsyncFunctionDef))}
    assert names and not names & {"compacted_bubbles", "pop_compacted_bubbles", "_bubbles_over", "_bubble_pop_nodes",
                                  "_list_sizes"}
