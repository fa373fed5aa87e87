"""The reads grouped by their path through the genes of interest without a GPU: hand-made cases with known answers (one
gene in two contexts at k = 3 and k = 5 with reads in both orientations; a read ending in the gene, assigned, ambiguous
or unassigned; two genes within k calls; a None window inside a run after filter_graph and after remove_node; a
palindromic key; a read wholly on marked windows; short reads, no ranks, unknown names, no reads, no edges), and the
product's numpy implementation (GeneMerGraph._gene_paths_over) against the loops of tests/gene_path_reference.py on
random reads and the fixtures, lazy graphs through the test double against host-edited graphs, and gene order."""
import os

import numpy as np
import pytest

from amira_b200 import construct_graph
from oracle import gmg_oracle as O
from tests.fake_device import OracleBackedDevice
from tests.gene_path_reference import gene_path_loop, marked_nodes, same_gene_paths
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES


@pytest.fixture(autouse=True)
def fake_device(monkeypatch):
    """lazy graphs on the test double, which has no gene_paths: served by the numpy implementation over its arrays"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", OracleBackedDevice)


def rc(read):
    return [("-" if g[0] == "+" else "+") + g[1:] for g in read[::-1]]


def expected(g, genes):
    """the loops over graph g: a lazy graph's device arrays, or a host-edited graph's objects"""
    if g._on_device():
        a = g._require_device_state().arrays()
        return gene_path_loop(a, marked_nodes(a, g._gene_ranks(list(genes))))
    amr = g.get_AMR_nodes(list(genes))
    return gene_path_loop(g._read_index_arrays(), [nh in amr for nh in g._nodes])


def paths(reads, k, genes):
    """gene_paths on a lazy graph, checked against the loops; the graph stays lazy"""
    g = construct_graph.GeneMerGraph(reads, k)
    x = g.gene_paths(genes)
    same_gene_paths(x, expected(g, genes))
    assert not reads or g.__dict__["_lazy"]
    return g, x


def span(g, genes, k):
    """the states of the windows of the gene list `genes` in graph g, found by the node keys"""
    rank = {n: i + 1 for i, n in enumerate(g._vocab.names)}
    ids = [(1 if x[0] == "+" else -1) * rank[x[1:]] for x in genes]
    keys = [tuple(r) for r in g._require_device_state().arrays()["node_key"].tolist()]
    out = []
    for i in range(len(ids) - k + 1):
        t = tuple(ids[i:i + k])
        r = tuple(-x for x in reversed(t))
        out.append(2 * keys.index(t) if t in keys else 2 * keys.index(r) + 1)
    return tuple(out)


def canon(s):
    r = tuple(x ^ 1 for x in reversed(s))
    return min(s, r)


def key(x, c):
    return tuple(x["key_state"][x["key_off"][c]:x["key_off"][c + 1]].tolist())


def members(x, c):
    return x["members"][x["member_off"][c]:x["member_off"][c + 1]].tolist()


A = ["+a%d" % i for i in range(1, 7)] + ["+amr"] + ["+b%d" % i for i in range(1, 7)]
B = ["+c%d" % i for i in range(1, 7)] + ["-amr"] + ["+d%d" % i for i in range(1, 7)]


@pytest.mark.parametrize("k", [3, 5])
def test_one_gene_in_two_contexts(k):
    reads = {"a0": A, "a1": A, "a2": rc(A), "b0": rc(B), "b1": B, "a3": A, "b2": rc(B)}
    g, x = paths(reads, k, ["amr"])
    assert x["occ_read"].tolist() == list(range(7)) and (x["occ_length"] == k).all() and (x["occ_flanks"] == 3).all()
    assert x["occ_win"].tolist() == [7 - k] * 7                       # the first window that holds the gene
    assert x["occ_cluster"].tolist() == [0, 0, 0, 1, 1, 0, 1]
    assert members(x, 0) == [0, 1, 2, 5] and members(x, 1) == [3, 4, 6] and x["n_complete"].tolist() == [4, 3]
    sa, sb = span(g, A[6 - k:7 + k], k), span(g, B[6 - k:7 + k], k)          # the gene's windows and one flank each side
    assert len(sa) == k + 2 and key(x, 0) == canon(sa) and key(x, 1) == canon(sb)
    oa = 1 if sa <= canon(sa) else -1
    ob = 1 if sb <= canon(sb) else -1
    assert x["occ_orient"].tolist() == [oa, oa, -oa, -ob, ob, oa, -ob]


def test_a_read_that_ends_in_the_gene():
    k = 3
    end = A[:7]                                                        # ... a6 amr: the run has no right flank
    bad = A[:4] + ["+x"] + A[5:7]                                      # an error in its left flank
    reads = {"a0": A, "a1": rc(A), "b0": B, "p0": end, "p1": rc(end), "p2": bad}
    g, x = paths(reads, k, ["amr"])
    part = x["occ_flanks"][3:].tolist()
    assert part == [1, 2, 1] and x["occ_cluster"].tolist() == [0, 0, 1, 0, 0, -1]
    assert x["occ_orient"][3] == -x["occ_orient"][4]
    assert members(x, 0) == [0, 1, 3, 4] and x["n_complete"].tolist() == [2, 1]
    # both contexts share the left side: the same partial read is ambiguous
    shared = A[:7] + B[7:]
    g, x = paths({"a0": A, "s0": shared, "p0": end}, k, ["amr"])
    assert x["occ_cluster"].tolist() == [0, 1, -2] and members(x, 0) == [0] and members(x, 1) == [1]


def test_two_genes_within_k_calls_are_one_run():
    k = 3
    read = A[:7] + ["+b1", "+amr2"] + A[7:]
    g, x = paths({"r0": read, "r1": rc(read)}, k, ["amr", "amr2"])
    assert x["occ_length"].tolist() == [k + 2, k + 2] and x["occ_cluster"].tolist() == [0, 0]
    g, x = paths({"r0": read}, k, ["amr"])                             # one gene: its own run
    assert x["occ_length"].tolist() == [k]


def test_a_none_window_splits_a_run():
    # filter_graph: the rare marked gene in the middle of a run (k = 1) goes, its window becomes None
    common = ["+a", "+b", "+amr1", "+amr2", "+amr3", "+c", "+d"]
    rare = ["+a", "+b", "+amr1", "+amrx", "+amr3", "+c", "+d"]
    genes = ["amr1", "amr2", "amr3", "amrx"]
    g = construct_graph.GeneMerGraph({"r%d" % i: common for i in range(3)} | {"e": rare}, 1)
    g.filter_graph(2, 1)
    x = g.gene_paths(genes)
    same_gene_paths(x, expected(g, genes))
    assert g.__dict__["_lazy"]
    assert x["occ_read"].tolist() == [0, 1, 2, 3, 3] and x["occ_win"][3:].tolist() == [2, 4]
    assert x["occ_flanks"][3:].tolist() == [1, 2] and x["occ_cluster"].tolist() == [0, 0, 0, 0, 0]
    # remove_node on the host: the middle window of a k = 3 run
    g = construct_graph.GeneMerGraph({"a0": A, "a1": A}, 3)
    g.remove_node(g.get_nodes_containing("amr")[1])                   # the gene's windows are consecutive nodes
    x = g.gene_paths(["amr"])
    same_gene_paths(x, expected(g, ["amr"]))
    assert not g._on_device()
    assert len(x["occ_read"]) == 4 and set(x["occ_length"].tolist()) == {1} and (x["occ_cluster"] == -1).all()


def test_a_palindromic_key():
    read = ["+p", "+amr", "-amr", "-p"]                                # its own reverse complement
    g, x = paths({"r0": read, "r1": read, "r2": ["+q"] + read[:3]}, 1, ["amr"])
    s = key(x, 0)
    assert s == tuple(x ^ 1 for x in reversed(s)) and len(x["key_off"]) == 2
    assert x["occ_orient"].tolist()[:2] == [1, 1] and x["occ_cluster"].tolist() == [0, 0, 0]


def test_a_read_wholly_on_marked_windows():
    k = 3
    whole = ["+amr1", "+amr2", "+amr1", "+amr3"]
    ctx = ["+x1", "+x2", "+x3", "+x4"] + whole + ["+y1", "+y2", "+y3", "+y4"]
    g, x = paths({"c": ctx, "w": whole, "w2": rc(whole)}, k, ["amr1", "amr2", "amr3"])
    assert x["occ_flanks"].tolist() == [3, 0, 0] and x["occ_cluster"].tolist() == [0, 0, 0]
    assert x["occ_orient"][1] == -x["occ_orient"][2] and members(x, 0) == [0, 1, 2]
    g, x = paths({"w": whole}, k, ["amr1", "amr2", "amr3"])           # no cluster to join
    assert x["occ_cluster"].tolist() == [-1] and len(x["key_off"]) == 1 and len(x["members"]) == 0


def test_degenerate_inputs():
    empty_keys = ("key_state", "n_complete", "members", "occ_read")
    for reads, k, genes in (({"s": ["+amr", "+a"]}, 3, ["amr"]),                       # short read
                            ({"a0": A}, 3, []),                                         # no ranks
                            ({"a0": A}, 3, ["nope", "nada"]),                           # unknown names
                            ({}, 3, ["amr"]),                                           # no reads
                            ({"e": A[4:7], "f": ["+amr"]}, 3, ["amr"])):                # no edges (one window each)
        g, x = paths(reads, k, genes)
        if len(reads) < 2:
            assert all(len(x[f]) == 0 for f in empty_keys) and x["key_off"].tolist() == [0], (reads, genes)
    g, x = paths({"a0": A}, 3, ["nope", "amr"])                      # unknown names are ignored
    assert x["occ_cluster"].tolist() == [0]
    g, x = paths({"e": A[4:7], "f": ["+amr"]}, 3, ["amr"])
    assert x["occ_flanks"].tolist() == [0] and x["occ_cluster"].tolist() == [-1]
    with pytest.raises(AssertionError, match="Strand information"):
        construct_graph.GeneMerGraph({"a0": A}, 3).gene_paths(["+amr"])


def test_numpy_against_the_loops_on_random_reads():
    n_assigned = n_ambiguous = n_clusters = 0
    for seed in range(300):
        rng = np.random.default_rng(71000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 30)), int(rng.integers(2, 9)), int(rng.integers(1, 16)))
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            dev = OracleBackedDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        ranks = sorted(set(rng.integers(1, len(vocab) + 1, int(rng.integers(0, 3))).tolist())) if len(vocab) else []
        for step in range(2):
            a = dev.arrays()
            marked = marked_nodes(a, ranks)
            want = gene_path_loop(a, marked)
            same_gene_paths(construct_graph.GeneMerGraph._gene_paths_over(a, marked), want, "seed %d" % seed)
            n_clusters += len(want["n_complete"])
            n_assigned += int(((want["occ_flanks"] != 3) & (want["occ_cluster"] >= 0)).sum())
            n_ambiguous += int((want["occ_cluster"] == -2).sum())
            flags = (rng.random(len(a["node_cov"])) < 0.2).astype(np.uint8)
            try:
                dev.remove_nodes(flags)
            except TypeError:
                break
    assert n_clusters > 200 and n_assigned > 50 and n_ambiguous > 5, (n_clusters, n_assigned, n_ambiguous)


@pytest.mark.parametrize("name", FIXTURES)
def test_numpy_against_the_loops_on_the_fixtures(name):
    from tests.helpers import load_input
    vocab, ids, off, ps, pe = load_input(name)
    rng = np.random.default_rng(len(name))
    for k in (1, 3, 5):
        try:
            dev = OracleBackedDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        a = dev.arrays()
        for ranks in ([1], sorted(set(rng.integers(1, len(vocab) + 1, 6).tolist()))):
            marked = marked_nodes(a, ranks)
            same_gene_paths(construct_graph.GeneMerGraph._gene_paths_over(a, marked), gene_path_loop(a, marked),
                            "%s k=%d" % (name, k))


def test_lazy_against_host_edited_and_gene_order():
    from amira_b200 import synth
    cfg = synth.CONFIGS["c2"]
    ids, off = synth.generate(cfg, 0, 1500)
    names = synth.vocabulary_names(cfg.vocab)
    reads = synth.to_read_dict(ids, off, names)
    genes = [names[r - 1] for r in synth._pool(cfg).amr.tolist()] + [names[10]]
    lazy, hst = construct_graph.GeneMerGraph(reads, 3), construct_graph.GeneMerGraph(reads, 3)
    for g in (lazy, hst):
        g.filter_graph(2, 1)
    hst._touch()
    x = lazy.gene_paths(genes)
    assert lazy.__dict__["_lazy"] and not hst._on_device()
    same_gene_paths(hst.gene_paths(genes), x, "host-edited")
    same_gene_paths(lazy.gene_paths(genes[::-1] + genes[:2]), x, "gene order")
    same_gene_paths(x, expected(lazy, genes))
    assert len(x["n_complete"]) > 5 and (x["occ_cluster"] >= 0).sum() > 50


def test_synth_keeps_its_amr_genes():
    from amira_b200 import synth
    for name in ("c2", "c5"):
        p = synth._pool(synth.CONFIGS[name])
        cfg = synth.CONFIGS[name]
        assert len(p.amr) == cfg.n_amr and len(set(p.amr.tolist())) == cfg.n_amr
        lo, hi = cfg.amr_copies
        assert ((p.amr_loci >= lo * cfg.n_genomes) & (p.amr_loci <= hi * cfg.n_genomes)).all()
        assert (np.isin(p.amr, np.abs(p.pool))).all()


UPSTREAM = os.environ.get("AMIRA_REFERENCE_ROOT", "/root/reference")


@pytest.mark.skipif(not os.path.isfile(os.path.join(UPSTREAM, "amira", "construct_graph.py")),
                    reason="upstream checkout not present")
def test_gene_path_methods_are_not_upstream_names():
    """bind_upstream overrides upstream's methods by name: the new methods must not replace one of upstream's"""
    import ast
    with open(os.path.join(UPSTREAM, "amira", "construct_graph.py")) as f:
        tree = ast.parse(f.read())
    cls = [c for c in tree.body if isinstance(c, ast.ClassDef) and c.name == "GeneMerGraph"]
    assert len(cls) == 1
    names = {f.name for f in cls[0].body if isinstance(f, (ast.FunctionDef, ast.AsyncFunctionDef))}
    assert names and not names & {"gene_paths", "_gene_paths_over"}
