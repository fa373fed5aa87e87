"""amira_gmg_unitig_links and amira_gmg_read_unitig_paths on the GPU against link_loop / read_path_loop (their
definitions restated as plain loops, tests/unitig_path_reference.py), array by array: random tiny graphs before and
after removals, the fixtures, synthetic inputs unfiltered, filtered and trimmed, a 200 000-node chain and circles, an
emptied graph; the cached results after filters and replayed resident builds (also over reads changed in place and a
k change); filter masks that survive the calls; the calls in any order; compacted_links / read_unitig_paths on a
lazy graph against the same calls on a host-edited graph."""
import itertools

import numpy as np
import pytest

from oracle import gmg_oracle as O
from tests.test_linear_walks_cpu import chain_input, circular_input
from tests.test_random_small_cpu import random_reads
from tests.test_unitig_paths_cpu import check_links, check_paths
from tests.test_unitigs_cpu import FIXTURES
from tests.unitig_path_reference import UnitigPathDevice, link_loop, read_path_loop
from tests.unitig_reference import unitig_loop

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dg():
    from amira_b200.device_graph import DeviceGraph
    g = DeviceGraph(0)
    yield g
    g.close()


def same_arrays(x, y, ctx=""):
    assert x.keys() == y.keys(), ctx
    for f in x:
        assert x[f].dtype == y[f].dtype, (ctx, f, x[f].dtype, y[f].dtype)
        assert np.array_equal(x[f], y[f]), (ctx, f)


def same_paths(dev, ref, ctx=""):
    """links and read paths of the device against the loops over the double's arrays"""
    x, y = dev.unitig_links(), ref.unitig_links()
    same_arrays(x, y, (ctx, "links"))
    p, q = dev.read_unitig_paths(), ref.read_unitig_paths()
    same_arrays(p, q, (ctx, "paths"))
    return x, p


def test_gpu_unitig_paths_random_tiny_graphs(dg):
    n = 0
    for seed in range(400):
        rng = np.random.default_rng(35000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = UnitigPathDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        dg.build(ids, off, k)
        same_paths(dg, ref, "seed %d" % seed)
        flags = (rng.random(ref.sizes()["nodes"]) < 0.3).astype(np.uint8)
        try:
            ref.remove_nodes(flags)
        except TypeError:                                      # multi-edge: the device refuses it too
            continue
        dg.remove_nodes(flags)
        same_paths(dg, ref, "seed %d after remove_nodes" % seed)
        n += 1
    assert n >= 250


@pytest.mark.parametrize("name", FIXTURES)
def test_gpu_unitig_paths_fixtures(dg, name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    for k in (1, 3, 5):
        try:
            ref = UnitigPathDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        dg.build(ids, off, k, ps, pe)
        same_paths(dg, ref, "%s k=%d" % (name, k))


SCALE = [("c2", 20000, 3), ("c2", 20000, 5), ("c3", 60000, 3), ("c3", 60000, 5)]


@pytest.mark.parametrize("cfg_name,n_reads,k", SCALE)
def test_gpu_unitig_paths_synthetic(dg, cfg_name, n_reads, k):
    """unfiltered (with the invariants), after filter_graph(3, 1), after remove_low_coverage_components(5), and
    remove_short_linear_paths(4) on the drop-in class, which stays lazy"""
    from amira_b200 import GeneMerGraph, synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    ref = UnitigPathDevice().build(ids, off, k)
    dg.build(ids, off, k)
    l, p = same_paths(dg, ref, "unfiltered")
    a = ref.arrays()
    u = unitig_loop(a)
    check_links(a, u, l)
    check_paths(a, u, p)
    same_paths(dg, ref, "unfiltered, cached")
    for g in (dg, ref):
        g.filter_graph(3, 1)
    same_paths(dg, ref, "filtered")
    for g in (dg, ref):
        g.remove_low_coverage_components(5)
    same_paths(dg, ref, "after remove_low_coverage_components")
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS[cfg_name].vocab))
    g = GeneMerGraph(reads, k)
    g.remove_short_linear_paths(4)
    got_l, got_p = g.compacted_links(), g.read_unitig_paths()
    assert g.__dict__["_lazy"]
    a = g._require_device_state().arrays()
    u = unitig_loop(a)
    same_arrays(got_l, link_loop(a, u), "links after remove_short_linear_paths")
    same_arrays(got_p, read_path_loop(a, u), "paths after remove_short_linear_paths")


def test_gpu_unitig_paths_chain_and_circle(dg):
    for (ids, off), k in ((chain_input(200000), 1), (circular_input(5000, 3), 3), (circular_input(5000, 1), 1)):
        ref = UnitigPathDevice().build(ids, off, k)
        dg.build(ids, off, k)
        l, p = same_paths(dg, ref, "%d genes k=%d" % (len(ids), k))
        assert len(l["edge"]) == 0 and p["path_off"].tolist() == [0, 1]


def test_gpu_unitig_paths_after_replayed_resident_builds(dg):
    """five replayed builds of a resident CSR; then the reads changed in place under the same pointers (the replayed
    graph builds another graph), then k = 5: the cached results of the earlier graph are not reused"""
    import torch
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 8000)
    d_ids, d_off = torch.from_numpy(ids.copy()).cuda(), torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    ref = UnitigPathDevice().build(ids, off, 3)
    for _ in range(5):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
        same_paths(dg, ref, "replayed")
    ids2 = np.ascontiguousarray(ids[::-1] * -1)                # every read's genes of another read, reversed
    d_ids.copy_(torch.from_numpy(ids2))
    torch.cuda.synchronize()
    for _ in range(2):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    same_paths(dg, UnitigPathDevice().build(ids2, off, 3), "reads changed in place")
    for _ in range(2):
        dg.build(d_ids, d_off, 5, on_device=True, wait=False)
    same_paths(dg, UnitigPathDevice().build(ids2, off, 5), "k = 5")


def test_gpu_unitig_paths_keep_filter_masks(dg):
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    ref = UnitigPathDevice().build(ids, off, 3)
    dg.build(ids, off, 3)
    for g in (dg, ref):
        g.filter_graph(3, 1)
    nk, ek = dg.filter_masks()
    assert not nk.all()
    same_paths(dg, ref)
    dg.linear_walks(np.arange(0, 2 * dg.sizes()["nodes"], 5))   # the walks' buffers beside these
    same_paths(dg, ref, "after linear_walks")
    x, y = dg.filter_masks()
    assert np.array_equal(x, nk) and np.array_equal(y, ek)


def test_gpu_unitig_paths_on_an_emptied_graph(dg):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input("synth_c2_2000")
    dg.build(ids, off, 3, ps, pe)
    dg.filter_graph(10**9, 1)
    assert dg.sizes()["nodes"] == 0
    l, p = dg.unitig_links(), dg.read_unitig_paths()
    assert all(len(l[f]) == 0 for f in l)
    assert p["path_off"].tolist() == [0] * (len(off)) and all(len(p[f]) == 0 for f in p if f != "path_off")
    ref = UnitigPathDevice().build(ids, off, 3, ps, pe)
    dg.build(ids, off, 3, ps, pe)
    same_paths(dg, ref, "rebuilt")


def test_gpu_unitig_paths_short_and_no_reads(dg):
    """all reads short, and no read at all: zero links, all-zero path_off"""
    reads = {"r1": ["+a", "+b"], "r2": ["+c"]}
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    dg.build(ids, off, 3)
    l, p = dg.unitig_links(), dg.read_unitig_paths()
    assert all(len(l[f]) == 0 for f in l) and p["path_off"].tolist() == [0, 0, 0]
    dg.build(np.zeros(0, np.int32), np.zeros(1, np.int64), 3)
    l, p = dg.unitig_links(), dg.read_unitig_paths()
    assert all(len(l[f]) == 0 for f in l) and p["path_off"].tolist() == [0]


def test_gpu_unitig_paths_call_order(dg):
    """unitigs, read paths, links and linear walks in any order give the same arrays; after one read_unitig_paths a
    repeated unitigs launches no kernel"""
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 4000)
    ref = UnitigPathDevice().build(ids, off, 3)
    want = {"unitigs": ref.unitigs(), "paths": ref.read_unitig_paths(), "links": ref.unitig_links()}
    calls = {"unitigs": lambda: dg.unitigs(), "paths": lambda: dg.read_unitig_paths(), "links": lambda: dg.unitig_links(),
             "walks": lambda: dg.linear_walks(np.arange(0, 2 * dg.sizes()["nodes"], 7))}
    walks = None
    for order in itertools.permutations(calls):
        dg.build(ids, off, 3)
        for name in order:
            got = calls[name]()
            if name == "walks":
                walks = got if walks is None else walks
                assert all(np.array_equal(x, y) for x, y in zip(got, walks)), order
            else:
                same_arrays(got, want[name], (order, name))
    dg.build(ids, off, 3)
    dg.read_unitig_paths()
    n = dg.kernel_launches()
    same_arrays(dg.unitigs(), want["unitigs"], "after read_unitig_paths")
    assert dg.kernel_launches() == n


@pytest.mark.parametrize("name,k", [("synth_c2_2000", 3), ("fixture_eight", 3), ("synth_c5_2000", 5)])
def test_gpu_links_and_paths_lazy_equal_host_path(name, k):
    """the device path leaves the graph lazy and gives the arrays the host path gives on a host-edited build of the
    same reads, also after filter_graph"""
    from amira_b200 import GeneMerGraph
    from tests.helpers import load_input, read_dict
    vocab, ids, off, ps, pe = load_input(name)
    reads, pos = read_dict(vocab, ids, off, ps, pe)
    for filt in (False, True):
        lazy = GeneMerGraph(reads, k, pos)
        host = GeneMerGraph(reads, k, pos)
        if filt:
            lazy.filter_graph(2, 1)
            host.filter_graph(2, 1)
        host._touch()
        got_l, got_p = lazy.compacted_links(), lazy.read_unitig_paths()
        assert lazy.__dict__["_lazy"]
        same_arrays(got_l, host.compacted_links(), (filt, "links"))
        same_arrays(got_p, host.read_unitig_paths(), (filt, "paths"))
