"""Unitigs without a GPU: the invariants of the compacted graph on unitig_loop (tests/unitig_reference.py, the reference
of the GPU tests) over random tiny graphs, the fixtures and hand-made probes (self edges, hairpins, tandem repeats);
the product's host implementation (GeneMerGraph._unitigs_over) against unitig_loop on lazy graphs through the test
double and on host-edited graphs, after filters and removals; a long chain and a circle."""
import os

import numpy as np
import pytest

from amira_b200 import construct_graph
from oracle import gmg_oracle as O
from tests.fake_device import OracleBackedDevice
from tests.test_linear_walks_cpu import chain_input, circular_input
from tests.test_random_small_cpu import random_reads
from tests.unitig_reference import UnitigDevice, unitig_loop, unitig_succ

FIXTURES = ["fixture_one", "fixture_three", "fixture_four", "fixture_five", "fixture_six", "fixture_seven",
            "fixture_eight", "fixture_nine"]
PROBES = [({"r1": ["+a", "+a", "+a", "+a", "+a"]}, (1, 2, 3)),
          ({"r1": ["+p", "+x", "+y", "-y", "-x", "-p"]}, (1, 2, 3)),
          ({"r1": ["+a", "-a", "+b"]}, (1,)),
          ({"r1": ["+g1", "+g2", "+g1", "+g2"], "r2": ["-g1", "-g2", "-g1", "-g2"]}, (1, 2, 3))]


@pytest.fixture
def fake_device(monkeypatch):
    """lazy graphs on the test double without unitigs(): compacted by the host implementation over its arrays"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", OracleBackedDevice)


def check_invariants(a, r):
    """the unitigs r of the graph arrays a: a partition of the nodes into maximal chains joined by internal edges"""
    N, E = len(a["node_cov"]), len(a["edge_src"])
    off, nodes = r["unitig_off"], r["unitig_nodes"]
    U = len(off) - 1
    assert off[0] == 0 and off[-1] == N and (np.diff(off) > 0).all()
    assert sorted(nodes.tolist()) == list(range(N))                                      # every node once
    unit = np.repeat(np.arange(U), np.diff(off))
    assert np.array_equal(r["node_unitig"][nodes], unit)
    assert np.array_equal(r["node_pos"][nodes], np.arange(N) - off[unit])
    # consecutive nodes (and the last and the first of a circular unitig) are joined both ways by internal edges
    internal = {(s, t) for s, t, f in zip(a["edge_src"].tolist(), a["edge_tgt"].tolist(), r["edge_internal"].tolist()) if f}
    for u in range(U):
        x = nodes[off[u]:off[u + 1]].tolist()
        pairs = list(zip(x, x[1:])) + ([(x[-1], x[0])] if r["circular"][u] else [])
        for p, q in pairs:
            assert (p, q) in internal and (q, p) in internal, (u, p, q)
    # the listed state of every node follows the successor rule; neither end of a linear unitig extends
    succ = unitig_succ(a)
    state = [2 * n + (r["node_orient"][n] == -1) for n in nodes.tolist()]
    for u in range(U):
        st = state[off[u]:off[u + 1]]
        assert all(succ[s] == t for s, t in zip(st, st[1:]))
        if r["circular"][u]:
            assert succ[st[-1]] == st[0]
        else:
            assert succ[st[-1]] == -1 and succ[st[0] ^ 1] == -1
    # ids by smallest node ascending, listed through that node's even state, a circular unitig from it
    first = np.asarray([nodes[off[u]:off[u + 1]].min() for u in range(U)], np.int64)
    assert (np.diff(first) > 0).all()
    assert (r["node_orient"][first] == 1).all()
    circ = np.flatnonzero(r["circular"])
    assert np.array_equal(nodes[off[circ]], first[circ])
    assert int(r["edge_internal"].sum()) == 2 * (N - (U - len(circ))) and len(r["edge_internal"]) == E
    cov = a["node_cov"].astype(np.int64)[nodes]
    if U:
        assert np.array_equal(r["cov_sum"], np.add.reduceat(cov, off[:-1]))
        assert np.array_equal(r["cov_min"], np.minimum.reduceat(cov, off[:-1]))
        assert np.array_equal(r["cov_max"], np.maximum.reduceat(cov, off[:-1]))


def same(x, y, ctx=""):
    assert x.keys() == y.keys(), ctx
    for f in x:
        assert x[f].dtype == y[f].dtype and np.array_equal(x[f], y[f]), (ctx, f)


def host_unitigs(a):
    g = construct_graph.GeneMerGraph.__new__(construct_graph.GeneMerGraph)
    return g._unitigs_over(a)


def checked(a):
    r = unitig_loop(a)
    check_invariants(a, r)
    same(host_unitigs(a), r)
    return r


@pytest.mark.parametrize("k", [1, 2, 3])
def test_unitig_invariants_on_random_tiny_graphs(k):
    n = n_circ = 0
    for seed in range(3000):
        if n == 300:
            break
        rng = np.random.default_rng(21000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            dev = UnitigDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        r = checked(dev.arrays())
        n_circ += int(r["circular"].sum())
        n += 1
    assert n == 300 and n_circ > 0


@pytest.mark.parametrize("name", FIXTURES)
def test_unitig_invariants_on_fixtures(name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    for k in (1, 3, 5):
        try:
            dev = UnitigDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        checked(dev.arrays())


def test_unitig_invariants_on_probes():
    seen = 0
    for reads, ks in PROBES:
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        for k in ks:
            try:
                dev = UnitigDevice().build(ids, off, k)
            except AssertionError:
                continue
            checked(dev.arrays())
            seen += 1
    assert seen >= 8


def test_unitigs_of_a_long_chain_and_a_circle():
    a = UnitigDevice().build(*chain_input(200000), 1).arrays()
    r = checked(a)
    assert len(r["circular"]) == 1 and not r["circular"][0] and r["edge_internal"].all()
    a = UnitigDevice().build(*circular_input(5000, 3), 3).arrays()
    r = checked(a)
    assert r["circular"].tolist() == [1] and r["unitig_nodes"][0] == 0 and r["node_orient"][0] == 1
    assert r["unitig_off"].tolist() == [0, 5000]


def test_empty_graph_has_no_unitigs(fake_device):
    g = construct_graph.GeneMerGraph({}, 3)
    r = g.compacted_unitigs()
    assert r["unitig_off"].tolist() == [0] and all(len(r[f]) == 0 for f in r if f != "unitig_off")


def test_compacted_unitigs_on_lazy_and_host_edited_graphs(fake_device):
    """lazy graph through the double (host implementation over its arrays) and a host-edited build of the same reads
    (host implementation over index arrays from its objects) against unitig_loop, after filter_graph,
    remove_short_linear_paths and remove_node; the lazy graph stays lazy"""
    steps = [[], [("filter_graph", (2, 1))], [("filter_graph", (2, 1)), ("remove_short_linear_paths", (4,))]]
    n = n_circ = 0
    for seed in range(200):
        rng = np.random.default_rng(23000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        k = int(rng.integers(1, 4))
        try:
            construct_graph.GeneMerGraph(reads, k)
        except AssertionError:
            continue
        try:
            for ops in steps:
                lazy, host = construct_graph.GeneMerGraph(reads, k), construct_graph.GeneMerGraph(reads, k)
                for g in (lazy, host):
                    for op, args in ops:
                        getattr(g, op)(*args)
                got = lazy.compacted_unitigs()
                assert lazy.__dict__["_lazy"] or not len(reads)
                a = lazy._require_device_state().arrays() if len(reads) else host._unitig_index_arrays()
                want = unitig_loop(a)
                same(got, want, (seed, ops))
                host._touch()                                  # edited on the host: compacted from its objects
                assert not host._on_device()
                same(host.compacted_unitigs(), want, (seed, ops, "host-edited"))
                n_circ += int(want["circular"].sum())
            # remove_node on the host: the objects are the only copy of the graph
            objs = list(host.get_nodes().values())
            for i in rng.choice(len(objs), min(len(objs), 2), replace=False).tolist():
                host.remove_node(objs[i])
        except TypeError:                                      # a removal meets a multi-edge, as upstream's does
            continue
        a = host._unitig_index_arrays()
        r = host.compacted_unitigs()
        same(r, unitig_loop(a), (seed, "remove_node"))
        check_invariants(a, r)
        n += 1
    assert n >= 100 and n_circ > 0, (n, n_circ)


UPSTREAM = os.environ.get("AMIRA_REFERENCE_ROOT", "/root/reference")


@pytest.mark.skipif(not os.path.isfile(os.path.join(UPSTREAM, "amira", "construct_graph.py")),
                    reason="upstream checkout not present")
def test_compacted_unitigs_is_not_an_upstream_name():
    """bind_upstream overrides upstream's methods by name: the new method must not replace one of upstream's"""
    import ast
    with open(os.path.join(UPSTREAM, "amira", "construct_graph.py")) as f:
        tree = ast.parse(f.read())
    cls = [c for c in tree.body if isinstance(c, ast.ClassDef) and c.name == "GeneMerGraph"]
    assert len(cls) == 1
    names = {f.name for f in cls[0].body if isinstance(f, (ast.FunctionDef, ast.AsyncFunctionDef))}
    assert names and "compacted_unitigs" not in names
