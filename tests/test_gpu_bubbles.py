"""amira_gmg_bubbles on the GPU against bubble_loop (its definition restated as a plain loop,
tests/bubble_reference.py), array by array: random tiny graphs and graphs of reads with gene-call errors before and
after removals, the fixtures, synthetic inputs unfiltered, filtered and trimmed; the cached result after replayed
resident builds (also over reads changed in place); an emptied graph; the call in any order with unitigs,
unitig_links and read_unitig_paths; filter masks that survive the call; pop_compacted_bubbles on a lazy graph against
the host-edited path."""
import itertools

import numpy as np
import pytest

from oracle import gmg_oracle as O
from tests.bubble_reference import BubbleDevice, bubble_loop
from tests.test_bubbles_cpu import check_bubbles, error_reads
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES
from tests.unitig_path_reference import read_path_loop
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


def same_bubbles(dev, ref, ctx=""):
    x = dev.bubbles()
    same_arrays(x, ref.bubbles(), ctx)
    return x


def test_gpu_bubbles_random_tiny_graphs(dg):
    n = n_bub = 0
    for seed in range(400):
        rng = np.random.default_rng(45000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14))) \
            if seed % 2 else error_reads(rng)
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = BubbleDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        dg.build(ids, off, k)
        n_bub += len(same_bubbles(dg, ref, "seed %d" % seed)["source"])
        flags = (rng.random(ref.sizes()["nodes"]) < 0.2).astype(np.uint8)
        try:
            ref.remove_nodes(flags)
        except TypeError:                                      # multi-edge: the device refuses it too
            continue
        dg.remove_nodes(flags)
        same_bubbles(dg, ref, "seed %d after remove_nodes" % seed)
        n += 1
    assert n >= 250 and n_bub >= 20


@pytest.mark.parametrize("name", FIXTURES)
def test_gpu_bubbles_fixtures(dg, name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    for k in (1, 3, 5):
        try:
            ref = BubbleDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        dg.build(ids, off, k, ps, pe)
        same_bubbles(dg, ref, "%s k=%d" % (name, k))


SCALE = [("c2", 20000, 3), ("c2", 20000, 5), ("c3", 60000, 3), ("c3", 60000, 5)]


@pytest.mark.parametrize("cfg_name,n_reads,k", SCALE)
def test_gpu_bubbles_synthetic(dg, cfg_name, n_reads, k):
    """unfiltered (with the invariants), cached, after filter_graph(3, 1), and after remove_short_linear_paths(4) on
    the drop-in class, which stays lazy"""
    from amira_b200 import GeneMerGraph, synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    ref = BubbleDevice().build(ids, off, k)
    dg.build(ids, off, k)
    bub = same_bubbles(dg, ref, "unfiltered")
    a = ref.arrays()
    u = unitig_loop(a)
    check_bubbles(a, u, read_path_loop(a, u), bub)
    assert len(bub["source"]) > 0
    same_bubbles(dg, ref, "unfiltered, cached")
    for g in (dg, ref):
        g.filter_graph(3, 1)
    same_bubbles(dg, ref, "filtered")
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS[cfg_name].vocab))
    g = GeneMerGraph(reads, k)
    g.remove_short_linear_paths(4)
    got = g.compacted_bubbles()
    assert g.__dict__["_lazy"]
    a = g._require_device_state().arrays()
    u = unitig_loop(a)
    same_arrays(got, bubble_loop(a, u, read_path_loop(a, u)), "after remove_short_linear_paths")


def test_gpu_bubbles_after_replayed_resident_builds(dg):
    import torch
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 8000)
    d_ids, d_off = torch.from_numpy(ids.copy()).cuda(), torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    ref = BubbleDevice().build(ids, off, 3)
    for _ in range(3):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
        same_bubbles(dg, ref, "replayed")
    ids2 = np.ascontiguousarray(ids[::-1] * -1)                # every read's genes of another read, reversed
    d_ids.copy_(torch.from_numpy(ids2))
    torch.cuda.synchronize()
    for _ in range(2):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    same_bubbles(dg, BubbleDevice().build(ids2, off, 3), "reads changed in place")


def test_gpu_bubbles_keep_filter_masks(dg):
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    ref = BubbleDevice().build(ids, off, 3)
    dg.build(ids, off, 3)
    for g in (dg, ref):
        g.filter_graph(3, 1)
    nk, ek = dg.filter_masks()
    assert not nk.all()
    same_bubbles(dg, ref)
    x, y = dg.filter_masks()
    assert np.array_equal(x, nk) and np.array_equal(y, ek)


def test_gpu_bubbles_on_an_emptied_graph(dg):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input("synth_c2_2000")
    dg.build(ids, off, 3, ps, pe)
    dg.filter_graph(10**9, 1)
    assert dg.sizes()["nodes"] == 0
    bub = dg.bubbles()
    assert bub["branch_off"].tolist() == [0] and all(len(bub[f]) == 0 for f in bub if f != "branch_off")
    dg.build(np.zeros(0, np.int32), np.zeros(1, np.int64), 3)
    assert dg.bubbles()["branch_off"].tolist() == [0]
    ref = BubbleDevice().build(ids, off, 3, ps, pe)
    dg.build(ids, off, 3, ps, pe)
    same_bubbles(dg, ref, "rebuilt")


def test_gpu_bubbles_call_order(dg):
    """unitigs, links, read paths and bubbles in every order give the same arrays"""
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 4000)
    ref = BubbleDevice().build(ids, off, 3)
    want = {"unitigs": ref.unitigs(), "links": ref.unitig_links(), "paths": ref.read_unitig_paths(),
            "bubbles": ref.bubbles()}
    calls = {"unitigs": dg.unitigs, "links": dg.unitig_links, "paths": dg.read_unitig_paths, "bubbles": dg.bubbles}
    for order in itertools.permutations(calls):
        dg.build(ids, off, 3)
        for name in order:
            same_arrays(calls[name](), want[name], (order, name))
    dg.build(ids, off, 3)
    dg.bubbles()
    n = dg.kernel_launches()
    same_arrays(dg.read_unitig_paths(), want["paths"], "after bubbles")
    same_arrays(dg.unitigs(), want["unitigs"], "after bubbles")
    assert dg.kernel_launches() == n


@pytest.mark.parametrize("name,k", [("synth_c2_2000", 3), ("synth_c4_3000", 3), ("synth_c5_2000", 5)])
def test_gpu_pop_lazy_equals_host_path(name, k):
    """pop_compacted_bubbles on a lazy graph (device bubbles, device removal, stays lazy) against a host-edited build
    of the same reads: the same hashes in the same order, then the same exported arrays and marked reads; also
    after filter_graph and with a gene of interest"""
    from amira_b200 import GeneMerGraph
    from tests.helpers import load_input, read_dict
    vocab, ids, off, ps, pe = load_input(name)
    reads, pos = read_dict(vocab, ids, off, ps, pe)
    for filt, genes in ((False, {}), (True, {}), (False, {vocab[0]})):
        lazy = GeneMerGraph(reads, k, pos)
        host = GeneMerGraph(reads, k, pos)
        if filt:
            lazy.filter_graph(2, 1)
            host.filter_graph(2, 1)
        host._touch()
        got = lazy.pop_compacted_bubbles(genes)
        assert lazy.__dict__["_lazy"]
        want = host.pop_compacted_bubbles(genes)
        assert got == want, (filt, genes)
        assert len(got) > 0 or filt or genes
        same_arrays(lazy.compacted_unitigs(), host.compacted_unitigs(), (filt, "unitigs after"))
        same_arrays(lazy.compacted_bubbles(), host.compacted_bubbles(), (filt, "bubbles after"))
        same_arrays(lazy.read_unitig_paths(), host.read_unitig_paths(), (filt, "paths after"))
        assert list(lazy.get_nodes()) == list(host.get_nodes())
        assert sorted(lazy.get_edges()) == sorted(host.get_edges())
        assert lazy.get_readNodes() == host.get_readNodes()
        assert lazy.get_reads_to_correct() == host.get_reads_to_correct()
