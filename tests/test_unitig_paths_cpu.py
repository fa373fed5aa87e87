"""Unitig links and read paths without a GPU: the invariants of both on link_loop / read_path_loop
(tests/unitig_path_reference.py, the reference of the GPU tests) over random tiny graphs, the fixtures and hand-made
reads (circles gone round more than once, reverse traversals, reads entering and leaving mid-unitig, tandem repeats,
self edges, hairpins, reads removed entirely, short reads); the product's host implementation
(GeneMerGraph._links_over / _read_paths_over) against the loops on lazy graphs through the test double and on
host-edited graphs, after filters and removals; a long chain and a circle."""
import os
from collections import Counter

import numpy as np
import pytest

from amira_b200 import construct_graph
from oracle import gmg_oracle as O
from tests.fake_device import OracleBackedDevice
from tests.test_linear_walks_cpu import chain_input, circular_input
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES, same
from tests.unitig_path_reference import UnitigPathDevice, link_loop, read_path_loop
from tests.unitig_reference import unitig_loop


@pytest.fixture
def fake_device(monkeypatch):
    """lazy graphs on the test double without the new calls: served by the host implementation over its arrays"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", OracleBackedDevice)


def host():
    return construct_graph.GeneMerGraph.__new__(construct_graph.GeneMerGraph)


def check_links(a, u, l):
    """one link per junction edge in edge order, between unitig ends, never on a circular unitig, with its twin"""
    junction = np.flatnonzero(u["edge_internal"] == 0)
    assert np.array_equal(l["edge"], junction)
    assert len(l["edge"]) == len(a["edge_src"]) - int(u["edge_internal"].sum())
    assert np.array_equal(l["cov"], a["edge_cov"][junction])
    ulen = np.diff(u["unitig_off"])
    src, tgt = a["edge_src"][junction], a["edge_tgt"][junction]
    assert np.array_equal(l["from_unitig"], u["node_unitig"][src]) and np.array_equal(l["to_unitig"], u["node_unitig"][tgt])
    last_from = u["node_pos"][src] == ulen[l["from_unitig"]] - 1
    first_from = u["node_pos"][src] == 0
    assert np.all(np.where(l["from_orient"] == 1, last_from, first_from))
    # a self edge is one directed record (the build does not expand it into two), so its reverse is not in the node's
    # entering list, which may continue the unitig: the entering end and the twin rule hold between distinct nodes
    x = src != tgt
    first_to = u["node_pos"][tgt] == 0
    last_to = u["node_pos"][tgt] == ulen[l["to_unitig"]] - 1
    assert np.all(np.where(l["to_orient"] == 1, first_to, last_to)[x])
    assert np.isin(l["from_orient"], (-1, 1)).all() and np.isin(l["to_orient"], (-1, 1)).all()
    assert not u["circular"][l["from_unitig"]].any() and not u["circular"][l["to_unitig"]].any()
    fu, fo, tu, to = l["from_unitig"][x].tolist(), l["from_orient"][x], l["to_unitig"][x].tolist(), l["to_orient"][x]
    assert Counter(zip(fu, fo.tolist(), tu, to.tolist())) == Counter(zip(tu, (-to).tolist(), fu, (-fo).tolist()))


def check_paths(a, u, p):
    """the steps of every read expand back into exactly its live window nodes, in order, each step at its own windows,
    maximal, with the window directions of its orientation; short reads have empty paths"""
    woff, wn, wd = a["win_off"], a["win_node"], a["win_dir"]
    R = len(woff) - 1
    off = p["path_off"]
    assert len(off) == R + 1 and off[0] == 0 and (np.diff(off) >= 0).all() and off[-1] == len(p["unitig"])
    for f in ("unitig", "orient", "pos", "win", "length"):
        assert len(p[f]) == off[-1], f
    assert (np.diff(off)[a["is_short"] != 0] == 0).all()
    uoff, unodes = u["unitig_off"].tolist(), u["unitig_nodes"].tolist()
    for r in range(R):
        nodes = wn[woff[r]:woff[r + 1]].tolist()
        dirs = wd[woff[r]:woff[r + 1]].tolist()
        got, prev = [], None
        for t in range(off[r], off[r + 1]):
            un, o, pos, w, ln = (int(p[f][t]) for f in ("unitig", "orient", "pos", "win", "length"))
            size, circ = uoff[un + 1] - uoff[un], u["circular"][un]
            assert ln >= 1 and (circ or 0 <= pos + o * (ln - 1) < size)
            for i in range(ln):
                q = pos + o * i
                n = unodes[uoff[un] + (q % size if circ else q)]
                assert nodes[w + i] == n and dirs[w + i] * u["node_orient"][n] == o, (r, t, i)
                got.append(n)
            if prev is not None and prev[3] + prev[4] == w:        # adjacent steps: the later one does not continue
                pu, po, ppos, _, pln = prev
                end = ppos + po * (pln - 1)
                nxt = (end + po) % size if circ else end + po
                assert not (pu == un and po == o and nxt == pos), (r, t)
            if prev is not None:
                assert w >= prev[3] + prev[4]
            prev = (un, o, pos, w, ln)
        assert got == [n for n in nodes if n >= 0], r


def checked(a):
    u = unitig_loop(a)
    l, p = link_loop(a, u), read_path_loop(a, u)
    check_links(a, u, l)
    check_paths(a, u, p)
    same(host()._links_over(a), l)
    same(host()._read_paths_over(a, a), p)
    return u, l, p


def build(reads, k):
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    return UnitigPathDevice().build(ids, off, k)


@pytest.mark.parametrize("k", [1, 2, 3])
def test_path_invariants_on_random_tiny_graphs(k):
    n = n_circ = n_removed = 0
    for seed in range(3000):
        if n == 200:
            break
        rng = np.random.default_rng(31000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        try:
            dev = build(reads, k)
        except AssertionError:                                 # palindromic window
            continue
        u, _, _ = checked(dev.arrays())
        n_circ += int(u["circular"].sum())
        flags = (rng.random(dev.sizes()["nodes"]) < 0.3).astype(np.uint8)
        try:
            dev.remove_nodes(flags)
        except TypeError:                                      # a removal meets a multi-edge
            continue
        checked(dev.arrays())
        n_removed += 1
        n += 1
    assert n == 200 and n_circ > 0 and n_removed > 0


@pytest.mark.parametrize("name", FIXTURES)
def test_path_invariants_on_fixtures(name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    for k in (1, 3, 5):
        try:
            dev = UnitigPathDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        checked(dev.arrays())


def steps_of(p, r):
    return [tuple(int(p[f][t]) for f in ("unitig", "orient", "pos", "win", "length"))
            for t in range(p["path_off"][r], p["path_off"][r + 1])]


def test_read_going_round_a_circle_three_times():
    """the smallest circle: two nodes cannot form one (a -> b and b -> a are one undirected edge entry)"""
    dev = build({"r1": ["+a", "+b", "+c"] * 3 + ["+a"], "r2": ["-b", "-a", "-c", "-b", "-a", "-c", "-b"]}, 1)
    u, l, p = checked(dev.arrays())
    assert u["circular"].tolist() == [1] and u["unitig_off"].tolist() == [0, 3] and len(l["edge"]) == 0
    (s,), (t,) = steps_of(p, 0), steps_of(p, 1)
    assert s[0] == 0 and s[3:] == (0, 10)                      # one step, longer than its unitig
    assert t[1] == -s[1] and t[3:] == (0, 7)                   # round the other way


def test_read_traversing_a_unitig_backwards_and_mid_unitig():
    reads = {"r1": ["+a", "+b", "+c", "+d", "+e"], "r2": ["-d", "-c", "-b"], "r3": ["+b", "+c", "+d"]}
    for k in (1, 2):
        dev = build(reads, k)
        u, _, p = checked(dev.arrays())
        assert len(u["circular"]) == 1
        ln = 5 - k + 1
        (s1,), (s2,), (s3,) = steps_of(p, 0), steps_of(p, 1), steps_of(p, 2)
        assert s1[4] == ln and s2[4] == s3[4] == 3 - k + 1
        assert s2[1] == -s1[1] and s3[1] == s1[1]              # backwards, forwards
        assert 0 < s3[2] < ln - 1 or k == 2                    # r3 enters and leaves inside the unitig


def test_tandem_repeats_revisit_one_unitig():
    dev = build({"r1": ["+a", "+b", "+c", "+x", "+a", "+b", "+c", "+y", "+a", "+b", "+c"]}, 1)
    u, l, p = checked(dev.arrays())
    s = steps_of(p, 0)
    assert [x[3] for x in s] == [0, 3, 4, 7, 8] and [x[4] for x in s] == [3, 1, 3, 1, 3]
    assert s[0][:3] == s[2][:3] == s[4][:3]                    # the same unitig, three separate visits
    assert len(l["edge"]) > 0


def test_self_edge_and_hairpin():
    for reads, ks in (({"r1": ["+a", "+a", "+a", "+a", "+a"]}, (1, 2, 3)),
                      ({"r1": ["+p", "+x", "+y", "-y", "-x", "-p"]}, (1, 2, 3)),
                      ({"r1": ["+a", "-a", "+b"]}, (1,))):
        for k in ks:
            try:
                dev = build(reads, k)
            except AssertionError:
                continue
            checked(dev.arrays())
    dev = build({"r1": ["+a", "+a", "+a", "+a"]}, 1)
    _, l, p = checked(dev.arrays())
    assert [x[4] for x in steps_of(p, 0)] == [1, 1, 1, 1]      # a self edge never continues a step
    assert len(l["edge"]) == 1                                 # one directed record


def test_read_removed_entirely_and_short_reads():
    reads = {"r1": ["+a", "+b", "+c", "+d"], "r2": ["+x", "+y", "+z"], "r3": ["+a"], "r4": ["+b", "+c"]}
    dev = build(reads, 2)
    a = dev.arrays()
    assert a["is_short"].tolist() == [0, 0, 1, 0]
    gone = np.zeros(dev.sizes()["nodes"], np.uint8)
    gone[a["win_node"][a["win_off"][1]:a["win_off"][2]]] = 1   # every node of r2
    dev.remove_nodes(gone)
    a = dev.arrays()
    _, _, p = checked(a)
    assert (a["win_node"][a["win_off"][1]:a["win_off"][2]] < 0).all()
    assert np.diff(p["path_off"]).tolist() == [1, 0, 0, 1]
    _, _, p = checked(build({"r1": ["+a", "+b"], "r2": ["+c"]}, 3).arrays())
    assert p["path_off"].tolist() == [0, 0, 0]


def test_paths_of_a_long_chain_and_a_circle():
    a = UnitigPathDevice().build(*chain_input(200000), 1).arrays()
    u, l, p = checked(a)
    assert p["path_off"].tolist() == [0, 1] and p["length"].tolist() == [200000] and len(l["edge"]) == 0
    a = UnitigPathDevice().build(*circular_input(5000, 3), 3).arrays()
    u, l, p = checked(a)
    assert u["circular"].tolist() == [1] and p["length"].tolist() == [5001] and len(l["edge"]) == 0


def test_empty_graph_has_no_links_and_no_paths(fake_device):
    g = construct_graph.GeneMerGraph({}, 3)
    l, p = g.compacted_links(), g.read_unitig_paths()
    assert all(len(l[f]) == 0 for f in l)
    assert p["path_off"].tolist() == [0] and all(len(p[f]) == 0 for f in p if f != "path_off")


def test_links_and_paths_on_lazy_and_host_edited_graphs(fake_device):
    """lazy graph through the double (host implementation over its arrays) and a host-edited build of the same reads
    (host implementation over index arrays from its objects and _readNodes) against the loops, after filter_graph,
    remove_low_coverage_components, remove_short_linear_paths and remove_node; the lazy graph stays lazy"""
    steps = [[], [("filter_graph", (2, 1))], [("remove_low_coverage_components", (3,))],
             [("filter_graph", (2, 1)), ("remove_short_linear_paths", (4,))]]
    n = n_none = 0
    for seed in range(200):
        rng = np.random.default_rng(33000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        k = int(rng.integers(1, 4))
        try:
            construct_graph.GeneMerGraph(reads, k)
        except AssertionError:
            continue
        try:
            for ops in steps:
                lazy, hst = construct_graph.GeneMerGraph(reads, k), construct_graph.GeneMerGraph(reads, k)
                for g in (lazy, hst):
                    for op, args in ops:
                        getattr(g, op)(*args)
                got_l, got_p = lazy.compacted_links(), lazy.read_unitig_paths()
                assert lazy.__dict__["_lazy"] or not len(reads)
                if len(reads):
                    a = lazy._require_device_state().arrays()
                    u = unitig_loop(a)
                    want_l, want_p = link_loop(a, u), read_path_loop(a, u)
                    same(got_l, want_l, (seed, ops))
                    same(got_p, want_p, (seed, ops))
                    n_none += int((a["win_node"] < 0).any())
                hst._touch()                                   # edited on the host: from its objects
                assert not hst._on_device()
                same(hst.compacted_links(), got_l, (seed, ops, "host-edited"))
                same(hst.read_unitig_paths(), got_p, (seed, ops, "host-edited"))
            objs = list(hst.get_nodes().values())
            for i in rng.choice(len(objs), min(len(objs), 2), replace=False).tolist():
                hst.remove_node(objs[i])
        except TypeError:                                      # a removal meets a multi-edge, as upstream's does
            continue
        a = hst._unitig_index_arrays()
        a.update(hst._read_index_arrays())
        u = unitig_loop(a)
        same(hst.compacted_links(), link_loop(a, u), (seed, "remove_node"))
        same(hst.read_unitig_paths(), read_path_loop(a, u), (seed, "remove_node"))
        a["is_short"] = np.zeros(len(a["win_off"]) - 1, np.uint8)
        check_links(a, u, hst.compacted_links())
        check_paths(a, u, hst.read_unitig_paths())
        n += 1
    assert n >= 100 and n_none > 0, (n, n_none)


UPSTREAM = os.environ.get("AMIRA_REFERENCE_ROOT", "/root/reference")


@pytest.mark.skipif(not os.path.isfile(os.path.join(UPSTREAM, "amira", "construct_graph.py")),
                    reason="upstream checkout not present")
def test_links_and_paths_are_not_upstream_names():
    """bind_upstream overrides upstream's methods by name: the new methods must not replace one of upstream's"""
    import ast
    with open(os.path.join(UPSTREAM, "amira", "construct_graph.py")) as f:
        tree = ast.parse(f.read())
    cls = [c for c in tree.body if isinstance(c, ast.ClassDef) and c.name == "GeneMerGraph"]
    assert len(cls) == 1
    names = {f.name for f in cls[0].body if isinstance(f, (ast.FunctionDef, ast.AsyncFunctionDef))}
    assert names and not names & {"compacted_links", "read_unitig_paths"}
