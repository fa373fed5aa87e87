"""amira_gmg_correct_bubble_reads on the GPU against correct_loop (its definition restated as a plain loop,
tests/bubble_correction_reference.py), array by array: random tiny graphs and graphs of reads with gene-call errors
before and after removals, the fixtures, synthetic inputs unfiltered, filtered and trimmed; device outputs against
host outputs; the rebuild from the corrected device CSR against the C oracle's build of its host copy; rounds of
correct -> rebuild that drop the old tensors; replayed resident builds; an emptied graph and a graph without bubbles;
bad replace_with; caches and filter masks that survive the call."""
import gc

import numpy as np
import pytest

from oracle import gmg_oracle as O
from tests.bubble_correction_reference import CorrectionDevice, replace_loop
from tests.test_bubbles_cpu import error_reads
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES
from tests.unitig_reference import unitig_loop

pytestmark = pytest.mark.gpu

FIELDS = ("ids", "off", "pos_start", "pos_end", "changed", "branch_rewritten")


@pytest.fixture(scope="module")
def dg():
    from amira_b200.device_graph import DeviceGraph
    g = DeviceGraph(0)
    yield g
    g.close()


def host(x):
    return {f: None if x[f] is None else x[f] if isinstance(x[f], np.ndarray) else x[f].cpu().numpy() for f in FIELDS}


def same_out(x, y, ctx=""):
    x, y = host(x), host(y)
    for f in FIELDS:
        if x[f] is None or y[f] is None:
            assert x[f] is None and y[f] is None, (ctx, f)
            continue
        assert x[f].dtype == y[f].dtype, (ctx, f, x[f].dtype, y[f].dtype)
        assert np.array_equal(x[f], y[f]), (ctx, f)


def random_replace(rng, bub):
    """per bubble a random kept branch; every other branch replaced or, at random, left alone"""
    off = bub["branch_off"].tolist()
    rw = np.full(off[-1], -1, np.int64)
    for b in range(len(off) - 1):
        keep = int(rng.integers(off[b], off[b + 1]))
        for g in range(off[b], off[b + 1]):
            if g != keep and rng.random() < 0.8:
                rw[g] = keep
    return rw


def same_correction(dev, ref, rw, ctx="", on_device=False):
    x = dev.correct_bubble_reads(rw, on_device=on_device)
    same_out(x, ref.correct_bubble_reads(rw), ctx)
    return x


def test_gpu_correction_random_tiny_graphs(dg):
    n = n_changed = 0
    for seed in range(400):
        rng = np.random.default_rng(48000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14))) \
            if seed % 2 else error_reads(rng)
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = CorrectionDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        dg.build(ids, off, k)
        x = same_correction(dg, ref, random_replace(rng, ref.bubbles()), "seed %d" % seed, on_device=seed % 3 == 0)
        n_changed += int(x["changed"].any())
        flags = (rng.random(ref.sizes()["nodes"]) < 0.2).astype(np.uint8)
        try:
            ref.remove_nodes(flags)
        except TypeError:                                      # multi-edge: the device refuses it too
            continue
        dg.remove_nodes(flags)
        same_correction(dg, ref, random_replace(rng, ref.bubbles()), "seed %d after remove_nodes" % seed)
        n += 1
    assert n >= 250 and n_changed >= 20, (n, n_changed)


@pytest.mark.parametrize("name", FIXTURES)
def test_gpu_correction_fixtures(dg, name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    rng = np.random.default_rng(7)
    for k in (1, 3, 5):
        try:
            ref = CorrectionDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        dg.build(ids, off, k, ps, pe)
        rw = random_replace(rng, ref.bubbles())
        same_correction(dg, ref, rw, "%s k=%d" % (name, k))
        same_correction(dg, ref, rw, "%s k=%d on device" % (name, k), on_device=True)


SCALE = [("c2", 20000, 3), ("c2", 20000, 5), ("c3", 60000, 3), ("c3", 60000, 5)]


@pytest.mark.parametrize("cfg_name,n_reads,k", SCALE)
def test_gpu_correction_synthetic(dg, cfg_name, n_reads, k):
    """unfiltered, after filter_graph(3, 1) and after filter_graph(1, 2), against the loop with the popping policy's
    replace_with; then correct_compacted_bubbles on a lazy graph trimmed by remove_short_linear_paths(4) against the
    same on a host-edited graph, and the rebuild from the device CSR against the oracle's build of its host copy"""
    from amira_b200 import GeneMerGraph, encode, synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    ref = CorrectionDevice().build(ids, off, k)
    dg.build(ids, off, k)
    for filt in (None, (3, 1), (1, 2)):
        if filt:
            ref.build(ids, off, k)
            dg.build(ids, off, k)
            for g in (dg, ref):
                g.filter_graph(*filt)
        u = unitig_loop(ref.arrays())
        bub = ref.bubbles()
        rw = replace_loop(u, bub, np.zeros(len(u["node_unitig"]), bool))
        x = same_correction(dg, ref, rw, (filt, "host outputs"))
        same_out(dg.correct_bubble_reads(rw, on_device=True), x, (filt, "device outputs"))
        assert filt or x["changed"].sum() > 0
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS[cfg_name].vocab))
    enc = encode.EncodedReads(reads)
    lazy, hst = GeneMerGraph(enc, k), GeneMerGraph(enc, k)
    for g in (lazy, hst):
        g.remove_short_linear_paths(4)
    hst._touch()
    e = lazy.correct_compacted_bubbles()
    assert lazy.__dict__["_lazy"] and e._device is not None
    e2 = hst.correct_compacted_bubbles()
    same_out({f: getattr(e, f) for f in FIELDS}, {f: getattr(e2, f) for f in FIELDS}, "lazy against host-edited")
    assert e2.reads == e.reads
    g2 = GeneMerGraph(e, k)
    assert O.diff_arrays(g2._require_device_state().arrays(), CorrectionDevice().build(e.ids, e.off, k).arrays()) == []


def test_gpu_correct_and_rebuild_rounds():
    """three rounds of correct_compacted_bubbles -> rebuild from the corrected resident CSR on C3, the previous
    reads dropped between rounds (a recycled offsets address meets the stale-count check of the resident build); each
    rebuild is bit-exact against the oracle's build of the corrected host copy, and the first round leaves fewer
    bubbles"""
    from amira_b200 import GeneMerGraph, encode, synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 20000)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS["c3"].vocab))
    g = GeneMerGraph(encode.EncodedReads(reads), 5)
    n_bub = [len(g.compacted_bubbles()["source"])]
    for _ in range(3):
        e = g.correct_compacted_bubbles()
        del g
        gc.collect()
        g = GeneMerGraph(e, 5)
        want = CorrectionDevice().build(e.ids, e.off, 5).arrays()
        del e
        gc.collect()
        assert O.diff_arrays(g._require_device_state().arrays(), want) == []
        n_bub.append(len(g.compacted_bubbles()["source"]))
    assert n_bub[1] < n_bub[0], n_bub


def test_gpu_correction_after_replayed_resident_builds(dg):
    import torch
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 8000)
    d_ids, d_off = torch.from_numpy(ids.copy()).cuda(), torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    ref = CorrectionDevice().build(ids, off, 3)
    rw = random_replace(np.random.default_rng(3), ref.bubbles())
    want = ref.correct_bubble_reads(rw)
    for _ in range(3):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
        same_out(dg.correct_bubble_reads(rw), want, "replayed")
        same_out(dg.correct_bubble_reads(rw, on_device=True), want, "replayed, on device")


def test_gpu_correction_without_bubbles(dg):
    """an emptied graph, an empty read set and a graph without bubbles: the output is the input, nothing changed"""
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input("synth_c2_2000")
    dg.build(ids, off, 3, ps, pe)
    dg.filter_graph(10**9, 1)
    assert dg.sizes()["nodes"] == 0
    for on_device in (False, True):
        x = host(dg.correct_bubble_reads(np.zeros(0, np.int64), on_device=on_device))
        assert np.array_equal(x["ids"], ids) and np.array_equal(x["off"], off) and not x["changed"].any()
        assert np.array_equal(x["pos_start"], ps) and np.array_equal(x["pos_end"], pe)
    dg.build(np.zeros(0, np.int32), np.zeros(1, np.int64), 3)
    x = dg.correct_bubble_reads(np.zeros(0, np.int64))
    assert x["off"].tolist() == [0] and len(x["ids"]) == 0 and len(x["changed"]) == 0
    reads = {"r%d" % i: ["+a", "+b", "+c", "+d", "+e"] for i in range(4)}
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    dg.build(ids, off, 3)
    x = dg.correct_bubble_reads(np.zeros(0, np.int64))
    assert np.array_equal(x["ids"], ids) and np.array_equal(x["off"], off) and not x["changed"].any()


def test_gpu_correction_bad_replace_with(dg):
    reads = {**{"t%d" % i: ["+a", "+b", "+c", "+d", "+e", "+f", "+g"] for i in range(5)},
             "e": ["+a", "+b", "+c", "+x", "+e", "+f", "+g"]}
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    dg.build(ids, off, 3)
    assert len(dg.bubbles()["branch_unitig"]) == 2
    for rw in ([-1, 1], [2, -1], [-2, 0], [-1], [0, 0]):
        with pytest.raises(ValueError):
            dg.correct_bubble_reads(np.asarray(rw))
    assert dg.correct_bubble_reads(np.asarray([-1, 0]))["changed"].tolist() == [0] * 5 + [1]


def test_gpu_correction_keeps_caches_and_filter_masks(dg):
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    ref = CorrectionDevice().build(ids, off, 3)
    dg.build(ids, off, 3)
    for g in (dg, ref):
        g.filter_graph(3, 1)
    nk, ek = dg.filter_masks()
    assert not nk.all()
    rw = random_replace(np.random.default_rng(5), ref.bubbles())
    dg.correct_bubble_reads(rw)                                # the first call reserves its buffers
    want = {"bubbles": dg.bubbles(), "unitigs": dg.unitigs(), "paths": dg.read_unitig_paths()}
    n = dg.kernel_launches()
    same_correction(dg, ref, rw, on_device=True)
    m = dg.kernel_launches()
    for name, f in (("bubbles", dg.bubbles), ("unitigs", dg.unitigs), ("paths", dg.read_unitig_paths)):
        x = f()
        assert all(np.array_equal(x[k], want[name][k]) for k in x), name
    assert dg.kernel_launches() == m and m > n
    x, y = dg.filter_masks()
    assert np.array_equal(x, nk) and np.array_equal(y, ek)
