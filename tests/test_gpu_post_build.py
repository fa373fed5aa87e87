"""The post-build half of the C ABI on the GPU -- the scans (read_length_coverages, node_coverage_stats,
junk_read_mask, nodes_containing, linear_steps) and the edits (remove_nodes, remove_nodes_without_reads_of) --
against the C-oracle test double, array by array, after every operation of a sequence: random tiny graphs, seeded
synthetic inputs at scale, nodes on 20000 reads, rounding ties, replayed builds and the empty graph."""
import numpy as np
import pytest

from oracle import gmg_oracle as O
from tests.fake_device import OracleBackedDevice
from tests.test_post_build_reference_cpu import ROUNDING_TIES, rounding_tie_mask, rounding_tie_reads
from tests.test_random_small_cpu import random_reads

pytestmark = pytest.mark.gpu

ERROR_RATES = (0.0, 0.2, 0.5, 0.7, 0.9, 1.0)
STEP_FIELDS = ("degree", "fw_next", "fw_dir", "fw_ext", "bw_next", "bw_dir", "bw_ext")


@pytest.fixture(scope="module")
def dg():
    from amira_b200.device_graph import DeviceGraph
    g = DeviceGraph(0)
    yield g
    g.close()


def thresholds(off):
    """16 read-length thresholds: 0, negative ones, small ones, the longest read, one more, 2^31 - 1"""
    longest = int(np.diff(off).max()) if len(off) > 1 else 0
    return np.array([0, -1, -(2**31), 1, 2, 3, 4, 5, 8, 13, 40, longest // 2, longest - 1, longest, longest + 1,
                     2**31 - 1], np.int32)


def rank_sets(ids, node_key, extra=()):
    """gene sets for nodes_containing / remove_nodes_without_reads_of: empty, duplicates, 0, V + 1, a gene of the
    input that is on no node (if there is one), and `extra`"""
    V = int(np.abs(ids).max()) if len(ids) else 1
    sets = [[], [1, 1, 1], [0], [V + 1], [0, V + 1, V, V, 1]] + [list(e) for e in extra]
    on_nodes = set(np.abs(node_key).ravel().tolist())
    absent = sorted(set(np.abs(ids).tolist()) - on_nodes)
    if absent:
        sets.append(absent[:1])
    return sets


class Pair:
    """the same graph on the device and on the test double; every operation is applied to both"""

    def __init__(self, dg, ids, off, k, ps=None, pe=None, ranks=()):
        self.dev, self.ref = dg, OracleBackedDevice()
        self.ids, self.off, self.extra_ranks = ids, off, ranks
        self.ref.build(ids, off, k, ps, pe)
        self.dev.build(ids, off, k, ps, pe)
        self.n_type_errors = 0

    def apply(self, op, *args):
        """-> True if the operation went through on both, False if both raised TypeError (multi-edge)"""
        errs = []
        for g in (self.dev, self.ref):
            try:
                getattr(g, op)(*args)
                errs.append(None)
            except TypeError:
                errs.append(TypeError)
        assert errs[0] == errs[1], (op, errs)
        self.n_type_errors += errs[0] is TypeError
        return errs[0] is None

    def check(self, ctx=""):
        """every export and every scan of the device equals the double's"""
        dev, ref = self.dev, self.ref
        b = ref.arrays()
        assert O.diff_arrays(dev.arrays(), b) == [], ctx
        got = []
        for g in (dev, ref):
            try:
                got.append(g.filter_masks())
            except RuntimeError:
                got.append(None)
        if got[1] is None:
            assert got[0] is None, (ctx, "filter masks of a call that did not complete or were overwritten")
        else:
            assert got[0] is not None, ctx
            for x, y in zip(got[0], got[1]):
                assert x.shape == y.shape and np.array_equal(x, y), ctx
        thr = thresholds(self.off)
        assert np.array_equal(dev.read_length_coverages(thr), ref.read_length_coverages(thr)), ctx
        assert dev.node_coverage_stats() == ref.node_coverage_stats(), ctx
        for er in ERROR_RATES:
            assert np.array_equal(dev.junk_read_mask(er), ref.junk_read_mask(er)), (ctx, er)
        for ranks in rank_sets(self.ids, b["node_key"], self.extra_ranks):
            assert np.array_equal(dev.nodes_containing(ranks), ref.nodes_containing(ranks)), (ctx, ranks)
        x, y = dev.linear_steps(), ref.linear_steps()
        for f in STEP_FIELDS:
            assert x[f].shape == y[f].shape and np.array_equal(x[f], y[f]), (ctx, f)
        return b

    def step(self, op, *args):
        ok = self.apply(op, *args)
        self.check("%s%r" % (op, args[:1] if op != "remove_nodes" else ()))
        return ok


def test_gpu_post_build_random_small_graphs(dg):
    """>= 300 tiny random read sets (multi-edges, self edges, hairpins, empty and short reads), each with a random
    sequence of 3..6 filters, component removals and node removals"""
    n_ops = {"filter_graph": 0, "remove_low_coverage_components": 0, "remove_nodes": 0,
             "remove_nodes_without_reads_of": 0}
    n_graphs = n_type_errors = 0
    for seed in range(400):
        rng = np.random.default_rng(7000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            p = Pair(dg, ids, off, k)
        except AssertionError:                               # palindromic window: covered by test_gpu_parity
            continue
        n_graphs += 1
        p.check("build seed %d" % seed)
        for _ in range(int(rng.integers(3, 7))):
            n = p.ref.sizes()["nodes"]
            op = ("filter_graph", "remove_low_coverage_components", "remove_nodes",
                  "remove_nodes_without_reads_of")[int(rng.integers(4))]
            if op == "filter_graph":
                args = (int(rng.integers(1, 4)), int(rng.integers(1, 4)))
            elif op == "remove_low_coverage_components":
                args = (int(rng.integers(1, 5)),)
            elif op == "remove_nodes":
                args = ((rng.random(n) < rng.choice([0.0, 0.1, 0.5, 1.0])).astype(np.uint8),)
            else:
                args = (rng.integers(0, len(vocab) + 2, int(rng.integers(0, 4))).astype(np.int32),)
            n_ops[op] += 1
            p.step(op, *args)
        n_type_errors += p.n_type_errors
    assert n_graphs >= 300 and min(n_ops.values()) >= 200 and n_type_errors > 0, (n_graphs, n_ops, n_type_errors)


SCALE = [("c2", 20000, 3, True), ("c3", 60000, 3, False), ("c3", 60000, 7, False), ("c5", 40000, 5, False),
         ("c3", 3000, 1, False)]


@pytest.mark.parametrize("cfg_name,n_reads,k,with_pos", SCALE)
def test_gpu_post_build_synthetic_chain(dg, cfg_name, n_reads, k, with_pos):
    """seeded synthetic inputs (many CTAs, positions with removals, k = 1 multi-edges): component removal, removal of
    every 7th node and every dead end, filter, pruning to the reads of a few genes -- compared after every step"""
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    ps = pe = None
    if with_pos:
        ps, pe = synth.positions_for(off, 7)
    counts = np.bincount(np.abs(ids))
    present = np.flatnonzero(counts)
    rare = int(present[np.argmin(counts[present])])
    common = int(present[np.argmax(counts[present])])
    p = Pair(dg, ids, off, k, ps, pe, ranks=[[rare], [common, rare]])
    p.check("build")
    p.step("remove_low_coverage_components", 5)
    flags = np.zeros(p.ref.sizes()["nodes"], np.uint8)
    flags[::7] = 1
    flags[p.ref.linear_steps()["degree"] == 1] = 1
    p.step("remove_nodes", flags)
    p.step("filter_graph", 3, 1)
    p.step("remove_nodes_without_reads_of", np.array([common, rare, int(present[len(present) // 2])], np.int32))
    if k == 1:
        assert p.n_type_errors > 0
    else:
        assert p.n_type_errors == 0 and p.ref.sizes()["nodes"] > 0


def test_gpu_post_build_heavy_nodes(dg):
    """nodes on 20000 reads (the per-warp loops over long read lists): pruning to the reads of a core gene keeps
    every node, pruning to a rare gene removes most of them"""
    from tests.test_gpu_parity import heavy_node_reads
    ids, off = heavy_node_reads()
    counts = np.bincount(np.abs(ids))
    present = np.flatnonzero(counts)
    rare = int(present[np.argmin(counts[present])])
    for k in (3, 5):
        p = Pair(dg, ids, off, k, ranks=[[1], [rare]])
        p.check("build k=%d" % k)
        n = p.ref.sizes()["nodes"]
        p.step("remove_nodes_without_reads_of", np.array([1], np.int32))
        assert p.ref.sizes()["nodes"] == n
        p.step("remove_nodes_without_reads_of", np.array([rare], np.int32))
        assert 0 < p.ref.sizes()["nodes"] < n // 10


@pytest.mark.parametrize("n,error_rate,want", ROUNDING_TIES)
def test_gpu_junk_read_mask_rounding_ties(dg, n, error_rate, want):
    """n * (1 - error_rate) on or next to .5: Python's round-half-even on the float64 product"""
    ids, off = rounding_tie_reads(n)
    p = Pair(dg, ids, off, 1)
    p.step("filter_graph", 2, 1)
    assert dg.junk_read_mask(error_rate).tolist() == rounding_tie_mask(n, want)


def test_gpu_scans_and_removal_after_replayed_builds(dg):
    """the same device-resident CSR built again and again without waiting (the library replays a captured CUDA
    graph), then the scans and a node removal straight away, before anything else looks at the graph"""
    import torch
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 8000)
    d_ids, d_off = torch.from_numpy(ids).cuda(), torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    ref = OracleBackedDevice().build(ids, off, 3)
    thr = thresholds(off)
    for rep in range(4):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    assert np.array_equal(dg.read_length_coverages(thr), ref.read_length_coverages(thr))
    for rep in range(3):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    assert dg.node_coverage_stats() == ref.node_coverage_stats()
    for rep in range(3):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    assert np.array_equal(dg.junk_read_mask(0.5), ref.junk_read_mask(0.5))
    for rep in range(3):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    x, y = dg.linear_steps(), ref.linear_steps()
    assert all(np.array_equal(x[f], y[f]) for f in STEP_FIELDS)
    for rep in range(3):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    flags = np.zeros(ref.sizes()["nodes"], np.uint8)
    flags[1::5] = 1
    dg.remove_nodes(flags)
    ref.remove_nodes(flags)
    assert O.diff_arrays(dg.arrays(), ref.arrays()) == []
    for rep in range(3):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
    ref.build(ids, off, 3)
    dg.remove_nodes_without_reads_of(np.array([5, 77], np.int32))
    ref.remove_nodes_without_reads_of(np.array([5, 77], np.int32))
    assert O.diff_arrays(dg.arrays(), ref.arrays()) == []
    for x, y in zip(dg.filter_masks(), ref.filter_masks()):
        assert np.array_equal(x, y)


def test_gpu_post_build_empty_graph(dg):
    """filter_graph removes every node; every scan, an empty remove_nodes and an AMR pruning then work on zero nodes,
    and the filter masks describe the last call; then a new build on the same handle"""
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input("synth_c2_2000")
    p = Pair(dg, ids, off, 3, ps, pe)
    n = p.ref.sizes()["nodes"]
    assert p.apply("filter_graph", 10**9, 1)
    nk, ek = dg.filter_masks()
    assert len(nk) == n and not nk.any() and not ek.any() and p.ref.sizes()["nodes"] == 0
    p.check("emptied")
    for op, args in (("remove_nodes", (np.zeros(0, np.uint8),)), ("filter_graph", (2, 1)),
                     ("remove_nodes_without_reads_of", (np.array([1, 2, 3], np.int32),)),
                     ("remove_low_coverage_components", (5,))):
        assert p.apply(op, *args)
        assert [len(m) for m in dg.filter_masks()] == [0, 0], op     # this call's masks, not the emptying filter's
        p.check(op)
    p = Pair(dg, ids, off, 3, ps, pe)
    p.check("rebuild")
    p.step("filter_graph", 3, 1)


def test_gpu_linear_steps_invalidate_the_filter_masks(dg):
    """linear_steps computes in the buffer of the last filter's edge mask: afterwards filter_masks() raises instead
    of handing out what is left in that buffer"""
    from amira_b200 import _lib, synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    p = Pair(dg, ids, off, 3)
    p.apply("filter_graph", 3, 1)
    nk, ek = dg.filter_masks()
    assert not nk.all() and not ek.all()
    dg.linear_steps()
    with pytest.raises(_lib.AmiraLibraryError):
        dg.filter_masks()
    assert p.apply("filter_graph", 4, 1)                     # the next filter has masks again
    assert len(dg.filter_masks()[0]) > 0
    p.check("second filter")


def test_gpu_failed_removal_leaves_graph_and_drops_masks(dg):
    """a removal that meets a multi-edge raises TypeError, changes nothing, leaves no filter masks behind, and the
    graph stays usable"""
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    p = Pair(dg, ids, off, 1)
    p.step("filter_graph", 2, 1)
    assert not p.apply("remove_nodes", np.ones(p.ref.sizes()["nodes"], np.uint8))
    p.check("after TypeError")
    with pytest.raises(RuntimeError):
        dg.filter_masks()


def test_gpu_class_removals_on_an_emptied_graph():
    """a materialised GeneMerGraph emptied by filter_graph: AMR pruning and dead-end removal leave it empty"""
    from amira_b200 import GeneMerGraph
    from tests.graph_snapshot import snapshot
    from tests.helpers import load_input, read_dict
    vocab, ids, off, ps, pe = load_input("synth_c2_2000")
    reads, pos = read_dict(vocab, ids, off, ps, pe)
    g = GeneMerGraph(reads, 3, pos)
    snapshot(g)
    assert not g.__dict__["_lazy"] and g.get_total_number_of_nodes() > 0
    g.filter_graph(10**9, 1)
    assert g.get_total_number_of_nodes() == 0
    g.remove_non_AMR_associated_nodes(vocab[:3])
    assert g.remove_short_linear_paths(4) == []
    assert g.get_total_number_of_nodes() == 0 and len(g.get_edges()) == 0
    assert all(all(n is None for n in nodes) for nodes in g.get_readNodes().values())
