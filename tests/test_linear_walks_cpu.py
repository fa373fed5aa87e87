"""Linear walks without a GPU: walk_loop and the double's linear_walks (tests/walk_reference.py, the reference of the GPU
tests) against GeneMerGraph._walk over the same step table, forward and backward, on random tiny graphs (self edges, multi-edges,
hairpins), a circular input and a long chain; and the index-array trimming policy of remove_short_linear_paths against
upstream's loop over host objects, on lazy and on host-edited graphs."""
import numpy as np
import pytest

from amira_b200 import construct_graph
from oracle import gmg_oracle as O
from tests.fake_device import OracleBackedDevice
from tests.graph_snapshot import snapshot
from tests.test_random_small_cpu import random_reads
from tests.walk_reference import WalkingDevice


@pytest.fixture(params=[WalkingDevice, OracleBackedDevice], ids=["with_walks", "step_table_only"])
def fake_device(monkeypatch, request):
    """the test double with linear_walks (the device graph's walks), and without (walked over its step table)"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", request.param)


def circular_input(n_genes, k):
    """one read around a circle of n_genes distinct genes, closed by its first k genes again -> (ids, off)"""
    ids = np.concatenate([np.arange(1, n_genes + 1), np.arange(1, k + 1)]).astype(np.int32)
    return ids, np.array([0, len(ids)], np.int64)


def chain_input(n_genes):
    ids = (np.arange(1, n_genes + 1) * np.where(np.arange(n_genes) % 3 == 1, -1, 1)).astype(np.int32)
    return ids, np.array([0, n_genes], np.int64)


def query_states(dev, rng, n_sample=2000):
    """every state of every degree-1 node, both states of the ends and the middle of the longest tip walk, and a
    seeded sample of the states"""
    deg = dev.linear_steps()["degree"]
    S = 2 * len(deg)
    tips = np.flatnonzero(deg == 1)
    tip_states = np.stack([2 * tips, 2 * tips + 1], 1).ravel()
    off, nodes = dev.linear_walks(tip_states)
    extra = []
    if len(tip_states):
        i = int(np.argmax(np.diff(off)))
        walk = nodes[off[i]:off[i + 1]]
        ends = [tip_states[i] >> 1] + ([int(walk[-1]), int(walk[len(walk) // 2])] if len(walk) else [])
        extra = [2 * e + s for e in ends for s in (0, 1)]
    sample = rng.integers(0, S, min(n_sample, S)) if S else np.zeros(0, np.int64)
    return np.concatenate([tip_states, np.asarray(extra, np.int64), sample]).astype(np.int64)


def walks_by_walk(g, st, states, want_branched):
    """_walk itself: forward from the state's side, and backward (reversed) from the same side"""
    out = []
    for s in states.tolist():
        side = "bw" if s & 1 else "fw"
        fw = g._walk(st, s >> 1, side, False, want_branched)
        if len(fw) < 5000:                                    # (the backward walk prepends: quadratic)
            bw = g._walk(st, s >> 1, side, True, want_branched)
            assert bw[-1] == s >> 1 and fw[1:] == bw[:-1][::-1]
        assert fw[0] == s >> 1
        out.append(fw[1:])
    return out


def check_walks(dev, states):
    g = construct_graph.GeneMerGraph.__new__(construct_graph.GeneMerGraph)
    st = {f: v.tolist() for f, v in dev.linear_steps().items()}
    for want in (False, True):
        off, nodes = dev.linear_walks(states, want)
        assert len(off) == len(states) + 1 and off[0] == 0
        got = [nodes[off[i]:off[i + 1]].tolist() for i in range(len(states))]
        assert got == walks_by_walk(g, st, np.asarray(states), want)


@pytest.mark.parametrize("k", [1, 2, 3])
def test_double_walks_equal_walk_on_random_tiny_graphs(k):
    n = 0
    for seed in range(3000):
        if n == 300:
            break
        rng = np.random.default_rng(9000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            dev = WalkingDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        S = 2 * dev.sizes()["nodes"]
        check_walks(dev, np.arange(S))
        n += 1
    assert n == 300


def test_double_walks_on_a_circle_and_a_long_chain():
    rng = np.random.default_rng(11)
    dev = WalkingDevice().build(*circular_input(5000, 3), 3)
    assert dev.sizes()["nodes"] == 5000 and (dev.linear_steps()["degree"] == 2).all()
    states = query_states(dev, rng, 200)
    off, _ = dev.linear_walks(states)
    assert (np.diff(off) == 4999).all()                       # around the circle, stopping before the start node
    check_walks(dev, states)
    dev = WalkingDevice().build(*chain_input(200000), 1)
    states = query_states(dev, rng, 20)
    off, _ = dev.linear_walks(states)
    assert np.diff(off).max() == 199999
    check_walks(dev, states)


def test_double_linear_walks_leave_filter_masks_and_reject_bad_states():
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 2000)
    dev = WalkingDevice().build(ids, off, 3)
    dev.filter_graph(2, 1)
    nk, ek = dev.filter_masks()
    S = 2 * dev.sizes()["nodes"]
    dev.linear_walks(np.arange(0, S, 7))
    assert all(np.array_equal(x, y) for x, y in zip(dev.filter_masks(), (nk, ek)))
    for bad in ([-1], [S], [0, S + 5]):
        with pytest.raises(ValueError):
            dev.linear_walks(bad)
    off0, nodes0 = dev.linear_walks([])
    assert off0.tolist() == [0] and len(nodes0) == 0


def upstream_remove_short_linear_paths(g, min_length, genes):
    """construct_graph.py:679-720 as upstream writes it, over the host objects of a graph edited on the host"""
    mean15 = g.get_mean_node_coverage() * 1.5 if g.get_nodes() else 0
    paths_to_remove = {}
    for node in list(g.get_nodes().values()):
        if g.get_degree(node) != 1:
            continue
        path = g.get_linear_path_for_node(node)
        if 0 < len(path) < min_length:
            if all(g.get_node_by_hash(n).get_node_coverage() > mean15 for n in path):
                continue
            paths_to_remove.setdefault(node.get_component(), []).append(path)
    AMR_nodes = g.get_AMR_nodes(genes)
    removed, seen = [], set()
    for component, paths in paths_to_remove.items():
        in_comp = {n.__hash__() for n in g.get_nodes_in_component(component)}
        for path in paths:
            if len(in_comp.intersection(path)) == len(in_comp):
                continue
            for nh in path:
                if nh in AMR_nodes or nh in seen:
                    continue
                seen.add(nh)
                removed.append(nh)
    for nh in removed:
        g.remove_node(g.get_node_by_hash(nh))
    return removed


def test_short_path_policy_on_lazy_and_host_edited_graphs(fake_device):
    """lazy device graph (arrays, linear_walks), host-edited graph (objects, _walk) and upstream's loop: the same
    list in the same order and the same graph afterwards; the lazy graph stays lazy"""
    n = n_removed = 0
    for seed in range(300):
        rng = np.random.default_rng(12000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        k = int(rng.integers(1, 4))
        genes = sorted({c[1:] for r in reads.values() for c in r})
        genes = [genes[int(i)] for i in rng.integers(0, len(genes), int(rng.integers(0, 3)))] if genes else []
        min_length = int(rng.integers(2, 8))
        try:
            lazy = construct_graph.GeneMerGraph(reads, k)
        except AssertionError:
            continue
        host = construct_graph.GeneMerGraph(reads, k)
        host._touch()
        ref = construct_graph.GeneMerGraph(reads, k)
        ref._touch()
        try:
            want = upstream_remove_short_linear_paths(ref, min_length, genes)
        except TypeError:                                     # remove_node meets a multi-edge
            continue
        assert lazy.remove_short_linear_paths(min_length, genes) == want
        assert lazy.__dict__["_lazy"] or not len(reads)
        assert host.remove_short_linear_paths(min_length, genes) == want
        assert snapshot(lazy) == snapshot(ref) == snapshot(host)
        n += 1
        n_removed += len(want) > 0
    assert n >= 200 and n_removed >= 20, (n, n_removed)
