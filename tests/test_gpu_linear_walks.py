"""amira_gmg_linear_walks on the GPU against walk_loop (GeneMerGraph._walk restated, tests/walk_reference.py), with and
without the branching node: all states of random tiny graphs and of the fixtures; tips, the longest chain and a seeded
sample of states on synthetic inputs, a 200 000-node chain and a circle; after filters, removals, replayed resident
builds (also over reads changed in place) and on an emptied graph.  And remove_short_linear_paths on a lazy graph
against the same call on a host-edited graph."""
import numpy as np
import pytest

from oracle import gmg_oracle as O
from tests.test_linear_walks_cpu import chain_input, circular_input, query_states
from tests.test_random_small_cpu import random_reads
from tests.walk_reference import WalkingDevice

pytestmark = pytest.mark.gpu

FIXTURES = ["fixture_one", "fixture_three", "fixture_four", "fixture_five", "fixture_six", "fixture_seven",
            "fixture_eight", "fixture_nine"]


@pytest.fixture(scope="module")
def dg():
    from amira_b200.device_graph import DeviceGraph
    g = DeviceGraph(0)
    yield g
    g.close()


def same_walks(dev, ref, states, ctx=""):
    for want in (False, True):
        x, y = dev.linear_walks(states, want), ref.linear_walks(states, want)
        assert x[0].dtype == np.int64 and x[1].dtype == np.int32, ctx
        assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]), (ctx, want)


def all_states(ref):
    return np.arange(2 * ref.sizes()["nodes"])


def test_gpu_linear_walks_random_tiny_graphs(dg):
    n = 0
    for seed in range(400):
        rng = np.random.default_rng(15000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = WalkingDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        dg.build(ids, off, k)
        same_walks(dg, ref, all_states(ref), "seed %d" % seed)
        flags = (rng.random(ref.sizes()["nodes"]) < 0.3).astype(np.uint8)
        try:
            ref.remove_nodes(flags)
        except TypeError:                                      # multi-edge: the device refuses it too
            continue
        dg.remove_nodes(flags)
        same_walks(dg, ref, all_states(ref), "seed %d after remove_nodes" % seed)
        n += 1
    assert n >= 250


@pytest.mark.parametrize("name", FIXTURES)
def test_gpu_linear_walks_fixtures(dg, name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    for k in (1, 3, 5):
        try:
            ref = WalkingDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        dg.build(ids, off, k, ps, pe)
        same_walks(dg, ref, all_states(ref), "%s k=%d" % (name, k))


SCALE = [("c2", 20000, 3), ("c3", 60000, 3), ("c3", 60000, 5)]


@pytest.mark.parametrize("cfg_name,n_reads,k", SCALE)
def test_gpu_linear_walks_synthetic(dg, cfg_name, n_reads, k):
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    ref = WalkingDevice().build(ids, off, k)
    dg.build(ids, off, k)
    rng = np.random.default_rng(k)
    same_walks(dg, ref, query_states(ref, rng), "unfiltered")
    for g in (dg, ref):
        g.remove_low_coverage_components(5)
        g.filter_graph(3, 1)
    same_walks(dg, ref, query_states(ref, rng), "filtered")
    flags = np.zeros(ref.sizes()["nodes"], np.uint8)
    flags[::11] = 1
    for g in (dg, ref):
        g.remove_nodes(flags)
    same_walks(dg, ref, query_states(ref, rng), "after remove_nodes")


def test_gpu_linear_walks_chain_and_circle(dg):
    rng = np.random.default_rng(5)
    for (ids, off), k in ((chain_input(200000), 1), (circular_input(5000, 3), 3), (circular_input(5000, 1), 1)):
        ref = WalkingDevice().build(ids, off, k)
        dg.build(ids, off, k)
        states = query_states(ref, rng, 20 if len(ids) > 10000 else 2000)
        same_walks(dg, ref, states, "%d genes k=%d" % (len(ids), k))


def test_gpu_linear_walks_after_replayed_resident_builds(dg):
    """five replayed builds of a resident CSR, then walks; the reads changed in place under the same pointers (the
    replayed graph builds another graph), then walks again: the jump table of the earlier graph is not reused"""
    import torch
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 8000)
    d_ids, d_off = torch.from_numpy(ids.copy()).cuda(), torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    rng = np.random.default_rng(1)
    ref = WalkingDevice().build(ids, off, 3)
    states = query_states(ref, rng)
    for _ in range(5):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    same_walks(dg, ref, states, "replayed")
    ids2 = np.ascontiguousarray(ids[::-1] * -1)                # every read's genes of another read, reversed
    d_ids.copy_(torch.from_numpy(ids2))
    torch.cuda.synchronize()
    for _ in range(2):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    ref2 = WalkingDevice().build(ids2, off, 3)
    same_walks(dg, ref2, query_states(ref2, rng), "reads changed in place")
    for _ in range(2):
        dg.build(d_ids, d_off, 5, on_device=True, wait=False)
    same_walks(dg, WalkingDevice().build(ids2, off, 5), states[states < 2 * dg.sizes()["nodes"]], "k = 5")


def test_gpu_linear_walks_keep_filter_masks_and_check_states(dg):
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    ref = WalkingDevice().build(ids, off, 3)
    dg.build(ids, off, 3)
    for g in (dg, ref):
        g.filter_graph(3, 1)
    nk, ek = dg.filter_masks()
    assert not nk.all()
    same_walks(dg, ref, all_states(ref))
    x, y = dg.filter_masks()
    assert np.array_equal(x, nk) and np.array_equal(y, ek)
    S = 2 * ref.sizes()["nodes"]
    for bad in ([-1], [S], [0, S], [2**31 - 1], [2**40], [-(2**40)]):
        with pytest.raises(ValueError):
            dg.linear_walks(bad)
    same_walks(dg, ref, [S - 1, 0, S - 1])                    # the handle stays usable
    off0, nodes0 = dg.linear_walks([])
    assert off0.tolist() == [0] and len(nodes0) == 0


def test_gpu_linear_walks_on_an_emptied_graph(dg):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input("synth_c2_2000")
    dg.build(ids, off, 3, ps, pe)
    dg.filter_graph(10**9, 1)
    assert dg.sizes()["nodes"] == 0
    for want in (False, True):
        off0, nodes0 = dg.linear_walks(np.zeros(0, np.int64), want)
        assert off0.tolist() == [0] and len(nodes0) == 0
    with pytest.raises(ValueError):
        dg.linear_walks([0])
    ref = WalkingDevice().build(ids, off, 3, ps, pe)
    dg.build(ids, off, 3, ps, pe)
    same_walks(dg, ref, all_states(ref), "rebuilt")


@pytest.mark.parametrize("name,k", [("synth_c2_2000", 3), ("fixture_eight", 3), ("synth_c5_2000", 5)])
def test_gpu_remove_short_linear_paths_lazy_equals_host_path(name, k):
    """the device path leaves the graph lazy, returns the same list in the same order as the host path over a
    second, host-edited build of the same reads, and leaves the same graph"""
    from amira_b200 import GeneMerGraph
    from tests.graph_snapshot import snapshot
    from tests.helpers import load_input, read_dict
    vocab, ids, off, ps, pe = load_input(name)
    reads, pos = read_dict(vocab, ids, off, ps, pe)
    genes = [vocab[i] for i in range(0, len(vocab), max(1, len(vocab) // 3))]
    n_removed = 0
    for min_length, gs in ((4, genes[:2]), (6, []), (12, genes)):
        lazy = GeneMerGraph(reads, k, pos)
        host = GeneMerGraph(reads, k, pos)
        host._touch()
        got = lazy.remove_short_linear_paths(min_length, gs)
        assert lazy.__dict__["_lazy"]
        want = host.remove_short_linear_paths(min_length, gs)
        assert got == want, (min_length, len(got), len(want))
        assert snapshot(lazy) == snapshot(host)
        n_removed += len(got)
    assert n_removed > 0
