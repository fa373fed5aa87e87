"""amira_gmg_unitigs on the GPU against unitig_loop (its definition restated as a plain loop, tests/unitig_reference.py),
array by array: random tiny graphs before and after removals, the fixtures, synthetic inputs unfiltered, filtered and
trimmed, a 200 000-node chain and circles, an emptied graph; the cached result after filters and replayed resident
builds (also over reads changed in place); filter masks that survive the call; compacted_unitigs on a lazy graph
against the same call on a host-edited graph."""
import numpy as np
import pytest

from oracle import gmg_oracle as O
from tests.test_linear_walks_cpu import chain_input, circular_input
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES, check_invariants
from tests.unitig_reference import UnitigDevice, unitig_loop

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dg():
    from amira_b200.device_graph import DeviceGraph
    g = DeviceGraph(0)
    yield g
    g.close()


def same_unitigs(dev, ref, ctx=""):
    x, y = dev.unitigs(), ref.unitigs()
    assert x.keys() == y.keys(), ctx
    for f in x:
        assert x[f].dtype == y[f].dtype, (ctx, f, x[f].dtype, y[f].dtype)
        assert np.array_equal(x[f], y[f]), (ctx, f)
    return x


def test_gpu_unitigs_random_tiny_graphs(dg):
    n = 0
    for seed in range(400):
        rng = np.random.default_rng(25000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = UnitigDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        dg.build(ids, off, k)
        same_unitigs(dg, ref, "seed %d" % seed)
        flags = (rng.random(ref.sizes()["nodes"]) < 0.3).astype(np.uint8)
        try:
            ref.remove_nodes(flags)
        except TypeError:                                      # multi-edge: the device refuses it too
            continue
        dg.remove_nodes(flags)
        same_unitigs(dg, ref, "seed %d after remove_nodes" % seed)
        n += 1
    assert n >= 250


@pytest.mark.parametrize("name", FIXTURES)
def test_gpu_unitigs_fixtures(dg, name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    for k in (1, 3, 5):
        try:
            ref = UnitigDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        dg.build(ids, off, k, ps, pe)
        same_unitigs(dg, ref, "%s k=%d" % (name, k))


SCALE = [("c2", 20000, 3), ("c2", 20000, 5), ("c3", 60000, 3), ("c3", 60000, 5)]


@pytest.mark.parametrize("cfg_name,n_reads,k", SCALE)
def test_gpu_unitigs_synthetic(dg, cfg_name, n_reads, k):
    """unfiltered, after filter_graph(3, 1) (the cached result of the unfiltered graph is not reused), after
    remove_low_coverage_components(5), and remove_short_linear_paths(4) on the drop-in class"""
    from amira_b200 import GeneMerGraph, synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    ref = UnitigDevice().build(ids, off, k)
    dg.build(ids, off, k)
    x = same_unitigs(dg, ref, "unfiltered")
    check_invariants(ref.arrays(), x)
    same_unitigs(dg, ref, "unfiltered, cached")
    for g in (dg, ref):
        g.filter_graph(3, 1)
    same_unitigs(dg, ref, "filtered")
    for g in (dg, ref):
        g.remove_low_coverage_components(5)
    same_unitigs(dg, ref, "after remove_low_coverage_components")
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS[cfg_name].vocab))
    g = GeneMerGraph(reads, k)
    g.remove_short_linear_paths(4)
    got = g.compacted_unitigs()
    assert g.__dict__["_lazy"]
    want = unitig_loop(g._require_device_state().arrays())
    for f in want:
        assert got[f].dtype == want[f].dtype and np.array_equal(got[f], want[f]), ("after remove_short_linear_paths", f)


def test_gpu_unitigs_chain_and_circle(dg):
    for (ids, off), k in ((chain_input(200000), 1), (circular_input(5000, 3), 3), (circular_input(5000, 1), 1)):
        ref = UnitigDevice().build(ids, off, k)
        dg.build(ids, off, k)
        x = same_unitigs(dg, ref, "%d genes k=%d" % (len(ids), k))
        assert len(x["circular"]) == 1


def test_gpu_unitigs_after_replayed_resident_builds(dg):
    """five replayed builds of a resident CSR; then the reads changed in place under the same pointers (the replayed
    graph builds another graph): the cached unitigs of the earlier graph are not reused"""
    import torch
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 8000)
    d_ids, d_off = torch.from_numpy(ids.copy()).cuda(), torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    for _ in range(5):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
        same_unitigs(dg, UnitigDevice().build(ids, off, 3), "replayed")
    ids2 = np.ascontiguousarray(ids[::-1] * -1)                # every read's genes of another read, reversed
    d_ids.copy_(torch.from_numpy(ids2))
    torch.cuda.synchronize()
    for _ in range(2):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    same_unitigs(dg, UnitigDevice().build(ids2, off, 3), "reads changed in place")
    for _ in range(2):
        dg.build(d_ids, d_off, 5, on_device=True, wait=False)
    same_unitigs(dg, UnitigDevice().build(ids2, off, 5), "k = 5")


def test_gpu_unitigs_keep_filter_masks(dg):
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    ref = UnitigDevice().build(ids, off, 3)
    dg.build(ids, off, 3)
    for g in (dg, ref):
        g.filter_graph(3, 1)
    nk, ek = dg.filter_masks()
    assert not nk.all()
    same_unitigs(dg, ref)
    dg.linear_walks(np.arange(0, 2 * dg.sizes()["nodes"], 5))   # the walks' buffers beside the unitigs'
    same_unitigs(dg, ref, "after linear_walks")
    x, y = dg.filter_masks()
    assert np.array_equal(x, nk) and np.array_equal(y, ek)


def test_gpu_unitigs_on_an_emptied_graph(dg):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input("synth_c2_2000")
    dg.build(ids, off, 3, ps, pe)
    dg.filter_graph(10**9, 1)
    assert dg.sizes()["nodes"] == 0
    x = dg.unitigs()
    assert x["unitig_off"].tolist() == [0] and all(len(x[f]) == 0 for f in x if f != "unitig_off")
    ref = UnitigDevice().build(ids, off, 3, ps, pe)
    dg.build(ids, off, 3, ps, pe)
    same_unitigs(dg, ref, "rebuilt")


@pytest.mark.parametrize("name,k", [("synth_c2_2000", 3), ("fixture_eight", 3), ("synth_c5_2000", 5)])
def test_gpu_compacted_unitigs_lazy_equals_host_path(name, k):
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
        got = lazy.compacted_unitigs()
        assert lazy.__dict__["_lazy"]
        want = host.compacted_unitigs()
        assert got.keys() == want.keys()
        for f in want:
            assert got[f].dtype == want[f].dtype and np.array_equal(got[f], want[f]), (filt, f)
