"""amira_gmg_clean_reads and clean_until_stable on the GPU against tests/clean_reference.py: the one pass against
clean_loop on random tiny graphs before and after removals, the fixtures, and C2 / C3 subsamples unfiltered, filtered
and trimmed with spared genes; the reductions to correct_bubble_reads and clip_tip_reads; the held-policy protocol and
bad host arrays; host against device outputs; caches and held policies that survive the call; the rebuild from the
device CSR against the C oracle; the rounds against clean_rounds_loop from lazy and host-edited graphs; the refusal of
a sharded handle."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import gmg_oracle as O
from tests.clean_reference import CleanDevice, clean_rounds_loop
from tests.test_bubbles_cpu import error_reads
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES

pytestmark = pytest.mark.gpu

FIELDS = ("ids", "off", "pos_start", "pos_end", "changed", "branch_rewritten", "tip_clipped")
CSR = ("ids", "off", "pos_start", "pos_end", "changed")


@pytest.fixture(scope="module")
def dg():
    from amira_b200.device_graph import DeviceGraph
    g = DeviceGraph(0)
    yield g
    g.close()


def host(x, fields=FIELDS):
    return {f: None if x[f] is None else x[f] if isinstance(x[f], np.ndarray) else x[f].cpu().numpy() for f in fields}


def same_out(x, y, ctx="", fields=FIELDS):
    x, y = host(x, fields), host(y, fields)
    for f in fields:
        if x[f] is None or y[f] is None:
            assert x[f] is None and y[f] is None, (ctx, f)
            continue
        assert x[f].dtype == y[f].dtype, (ctx, f, x[f].dtype, y[f].dtype)
        assert np.array_equal(x[f], y[f]), (ctx, f)


def same_clean(dev, ref, min_tip_length, ranks=(), ctx="", on_device=False):
    """both policies, then the pass with the held policies; returns the device output"""
    assert dev.bubble_policy(ranks) == ref.bubble_policy(ranks), (ctx, "bubble policy")
    assert dev.tip_policy(min_tip_length, ranks) == ref.tip_policy(min_tip_length, ranks), (ctx, "tip policy")
    x = dev.clean_reads(None, None, on_device=on_device)
    same_out(x, ref.clean_reads(None, None), ctx)
    return x


def test_gpu_clean_random_tiny_graphs(dg):
    n = n_both = 0
    for seed in range(400):
        rng = np.random.default_rng(56000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14))) \
            if seed % 2 else error_reads(rng, int(rng.integers(10, 40)))
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = CleanDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        dg.build(ids, off, k)
        ranks = [int(rng.integers(1, len(vocab) + 1))] if seed % 3 == 0 and len(vocab) else []
        min_tip_length = int(rng.integers(1, k + 4))
        x = host(same_clean(dg, ref, min_tip_length, ranks, "seed %d" % seed, on_device=seed % 3 == 1))
        n_both += int(x["branch_rewritten"].any() and x["tip_clipped"].any())
        flags = (rng.random(ref.sizes()["nodes"]) < 0.2).astype(np.uint8)
        try:
            ref.remove_nodes(flags)
        except TypeError:                                      # multi-edge: the device refuses it too
            continue
        dg.remove_nodes(flags)
        same_clean(dg, ref, min_tip_length, ranks, "seed %d after remove_nodes" % seed)
        n += 1
    assert n >= 250 and n_both >= 10, (n, n_both)


@pytest.mark.parametrize("name", FIXTURES)
def test_gpu_clean_fixtures(dg, name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    for k in (1, 3, 5):
        try:
            ref = CleanDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        dg.build(ids, off, k, ps, pe)
        same_clean(dg, ref, k + 1, (), "%s k=%d" % (name, k))
        same_clean(dg, ref, k + 1, (), "%s k=%d on device" % (name, k), on_device=True)


SCALE = [("c2", 20000, 3), ("c3", 20000, 5)]


@pytest.mark.parametrize("cfg_name,n_reads,k", SCALE)
def test_gpu_clean_synthetic(dg, cfg_name, n_reads, k):
    """unfiltered, after filter_graph(3, 1) and filter_graph(4, 6), against the loop with spared ranks, host and device
    outputs alike; then clean_compacted_reads on a lazy graph trimmed by remove_short_linear_paths(4) against the same
    on a host-edited graph"""
    from amira_b200 import GeneMerGraph, encode, synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    ref = CleanDevice().build(ids, off, k)
    for filt in (None, (3, 1), (4, 6)):
        ref.build(ids, off, k)
        dg.build(ids, off, k)
        if filt:
            for g in (dg, ref):
                g.filter_graph(*filt)
        x = same_clean(dg, ref, k + 1, (3, 7), (filt, "host outputs"))
        same_out(dg.clean_reads(None, None, on_device=True), x, (filt, "device outputs"))
        hx = host(x)
        assert filt or (hx["branch_rewritten"].sum() > 0 and hx["tip_clipped"].sum() > 0)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS[cfg_name].vocab))
    enc = encode.EncodedReads(reads)
    lazy, hst = GeneMerGraph(enc, k), GeneMerGraph(enc, k)
    for g in (lazy, hst):
        g.remove_short_linear_paths(4)
    hst._touch()
    e = lazy.clean_compacted_reads(k + 1)
    assert lazy.__dict__["_lazy"] and e._device is not None
    e2 = hst.clean_compacted_reads(k + 1)
    same_out({f: getattr(e, f) for f in FIELDS}, {f: getattr(e2, f) for f in FIELDS}, "lazy against host-edited")
    assert e2.reads == e.reads


def test_gpu_reductions_to_the_single_calls(dg):
    """all -1 replace_with gives clip_tip_reads, an all-zero clip gives correct_bubble_reads, field by field"""
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 20000)
    dg.build(ids, off, 5)
    _, rw = dg.bubble_policy((), want_replace_with=True)
    _, clip = dg.tip_policy(6, (), want_clip=True)
    x = dg.clean_reads(np.full(len(rw), -1), clip)
    same_out(x, dg.clip_tip_reads(clip), "no edits", CSR + ("tip_clipped",))
    assert not x["branch_rewritten"].any() and x["changed"].any()
    x = dg.clean_reads(rw, np.zeros(len(clip), np.uint8))
    same_out(x, dg.correct_bubble_reads(rw), "no clips", CSR + ("branch_rewritten",))
    assert not x["tip_clipped"].any() and x["changed"].any()
    both = host(dg.clean_reads(rw, clip))
    assert (both["changed"] >= x["changed"]).all() and both["changed"].sum() > x["changed"].sum()


def test_gpu_clean_protocol(dg):
    """AMIRA_E_STATE without a fresh held policy of either kind (after a build, a filter, a removal of no node, an
    overwrite by a host array); AMIRA_E_ARG for bad host arrays, checked before any device work"""
    from amira_b200 import _lib, synth
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 3000)
    L, n = dg._lib, C.c_int64()
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    call = lambda rw=None, clip=None: L.amira_gmg_clean_reads(dg._h, p(rw), p(clip), C.byref(n), *[None] * 7, 0)

    def fresh():
        dg.bubble_policy()
        dg.tip_policy(4)
        assert call() == _lib.OK

    dg.build(ids, off, 3)
    NB, Q = dg.bubble_counts()[1], dg.tip_count()
    assert NB > 0 and Q > 0
    assert call() == _lib.E_STATE
    dg.bubble_policy()
    assert call() == _lib.E_STATE                              # no tip policy
    dg.build(ids, off, 3)
    dg.tip_policy(4)
    assert call() == _lib.E_STATE                              # no bubble policy
    fresh()
    dg.remove_nodes(np.zeros(dg.sizes()["nodes"], np.uint8))   # a removal of no node is a new graph
    NB, Q = dg.bubble_counts()[1], dg.tip_count()
    assert call() == _lib.E_STATE
    fresh()
    assert call(np.full(NB, -1, np.int32)) == _lib.OK          # host replace_with overwrites the held one
    assert call() == _lib.E_STATE and call(None, np.zeros(Q, np.uint8)) == _lib.E_STATE
    fresh()
    assert call(None, np.zeros(Q, np.uint8)) == _lib.OK        # host flags overwrite the held ones
    assert call() == _lib.E_STATE
    fresh()
    bad_rw = np.full(NB, -1, np.int32)
    bad_rw[0] = 0                                              # a branch replaced by itself
    bad_clip = np.zeros(Q, np.uint8)
    bad_clip[Q // 2] = 2
    assert call(bad_rw) == _lib.E_ARG and call(None, bad_clip) == _lib.E_ARG
    assert call() == _lib.OK                                   # the refusals left both held policies
    for args in ((bad_rw, None), (None, bad_clip), (np.full(NB + 1, -1), None), (None, np.zeros(Q + 1, np.uint8))):
        with pytest.raises(ValueError):
            dg.clean_reads(*args)
    dg.filter_graph(2, 1)                                      # a new graph: both policies are gone
    if dg.bubble_counts()[1] or dg.tip_count():
        assert call() == _lib.E_STATE


def test_gpu_clean_keeps_caches_held_policies_and_filter_masks(dg):
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    ref = CleanDevice().build(ids, off, 3)
    dg.build(ids, off, 3)
    for g in (dg, ref):
        g.filter_graph(3, 1)
    nk, ek = dg.filter_masks()
    assert not nk.all()
    x = same_clean(dg, ref, 4)                                 # the first calls reserve the buffers
    want = {"tips": dg.tips(), "bubbles": dg.bubbles(), "unitigs": dg.unitigs(), "paths": dg.read_unitig_paths()}
    n = dg.kernel_launches()
    same_out(dg.clean_reads(None, None, on_device=True), x, "repeat")
    m = dg.kernel_launches()
    for name, f in (("tips", dg.tips), ("bubbles", dg.bubbles), ("unitigs", dg.unitigs), ("paths", dg.read_unitig_paths)):
        y = f()
        assert all(np.array_equal(y[k], want[name][k]) for k in y), name
    assert dg.kernel_launches() == m and m > n
    same_out(dg.correct_bubble_reads(None), ref.correct_bubble_reads(None), "held bubble policy",
             CSR + ("branch_rewritten",))
    same_out(dg.clip_tip_reads(None), ref.clip_tip_reads(None), "held tip policy", CSR + ("tip_clipped",))
    x, y = dg.filter_masks()
    assert np.array_equal(x, nk) and np.array_equal(y, ek)


def test_gpu_clean_on_empty_graphs(dg):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input("synth_c2_2000")
    dg.build(ids, off, 3, ps, pe)
    dg.filter_graph(10**9, 1)
    assert dg.bubble_policy() == 0 and dg.tip_policy(4) == 0
    for on_device in (False, True):
        x = host(dg.clean_reads(None, None, on_device=on_device))
        assert np.array_equal(x["ids"], ids) and np.array_equal(x["off"], off) and not x["changed"].any()
        assert np.array_equal(x["pos_start"], ps) and np.array_equal(x["pos_end"], pe)
    dg.build(np.zeros(0, np.int32), np.zeros(1, np.int64), 3)
    x = dg.clean_reads(None, None)
    assert x["off"].tolist() == [0] and len(x["ids"]) == 0 and len(x["changed"]) == 0


def test_gpu_rebuild_from_the_device_csr_with_its_call_count(dg):
    """the cleaned device CSR rebuilt with n_calls on the handle is bit-exact against the oracle's build of the host
    copy, and holds fewer bubbles and tips"""
    from amira_b200 import synth
    from amira_b200.device_graph import DeviceGraph
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 20000)
    dg.build(ids, off, 5)
    before = (dg.bubble_counts()[0], dg.tip_count())
    dg.bubble_policy()
    dg.tip_policy(6)
    x = dg.clean_reads(None, None, on_device=True)
    h2 = DeviceGraph(0)
    h2.build(x["ids"], x["off"], 5, on_device=True, n_calls=len(x["ids"]))
    hx = host(x)
    want = CleanDevice().build(hx["ids"], hx["off"], 5).arrays()
    assert O.diff_arrays(h2.arrays(), want) == []
    assert h2.bubble_counts()[0] < before[0] and h2.tip_count() < before[1]
    h2.close()


@pytest.mark.parametrize("filt", [None, (1, 2)])
def test_gpu_clean_until_stable(filt):
    """clean_until_stable against its definition from a lazy and a host-edited graph; the final graph against the
    oracle's build of the final reads"""
    from amira_b200 import GeneMerGraph, encode, synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 6000)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS["c3"].vocab))
    enc = encode.EncodedReads(reads)
    lazy, hst = GeneMerGraph(enc, 5), GeneMerGraph(enc, 5)
    hst._touch()
    results = []
    for g in (lazy, hst):
        graph, out = g.clean_until_stable(6, 30, {}, filt)
        want_g, want_e, want_changed, want_rounds = clean_rounds_loop(g, 6, 30, {}, filt, fast=True)
        assert out.rounds == want_rounds and len(out.rounds) >= 2
        assert out.reads == want_e.reads and np.array_equal(out.ids, want_e.ids) and np.array_equal(out.off, want_e.off)
        assert np.array_equal(out.changed, want_changed)
        assert np.array_equal(out.branch_rewritten, want_e.branch_rewritten)
        assert np.array_equal(out.tip_clipped, want_e.tip_clipped)
        assert graph.__dict__["_lazy"]
        ref = CleanDevice().build(out.ids, out.off, 5)
        if filt:
            ref.filter_graph(*filt)
        assert O.diff_arrays(graph._require_device_state().arrays(), ref.arrays()) == []
        results.append(out)
    assert results[0].reads == results[1].reads and results[0].rounds == results[1].rounds


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def test_gpu_clean_refuses_a_sharded_handle():
    n = _n_gpus()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    from tests.helpers import ROOT
    from tests.test_sharded import _free_port
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "sharded_clean_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0 and "SHARDED_CLEAN OK" in res.stdout, (res.stdout[-3000:], res.stderr[-3000:])
