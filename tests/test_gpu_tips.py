"""amira_gmg_tips, amira_gmg_tip_policy and amira_gmg_clip_tip_reads on the GPU against the loops of
tests/tip_reference.py, array by array: random tiny graphs before and after removals, with random min_length and
spared ranks; the fixtures; synthetic inputs unfiltered, filtered and trimmed; host clip flags against the device-held
policy; the refusals (no policy, a bad flag, a sharded handle); a junction with more than 32 tips; replayed resident
builds; an emptied graph and an empty read set; caches and filter masks that survive the calls; tip and bubble calls
interleaved on one graph; lazy against host-edited graphs; the rebuild from the clipped device CSR against the C
oracle's build of its host copy."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import gmg_oracle as O
from tests.test_bubbles_cpu import TRUE, error_reads
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES
from tests.tip_reference import TipPolicyDevice

pytestmark = pytest.mark.gpu

FIELDS = ("ids", "off", "pos_start", "pos_end", "changed", "tip_clipped")
TIP_FIELDS = ("tip_unitig", "tip_orient", "tip_attach", "tip_reads")


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


def same_tips(dev, ref, min_length, ranks=(), ctx="", on_device=False):
    """tips, the policy (count and flags) and the clip with the device-held flags; returns the clip output"""
    same_out(dev.tips(), ref.tips(), ctx, TIP_FIELDS)
    n, clip = dev.tip_policy(min_length, ranks, want_clip=True)
    m, want = ref.tip_policy(min_length, ranks, want_clip=True)
    assert n == m and np.array_equal(clip, want), (ctx, "policy")
    x = dev.clip_tip_reads(None, on_device=on_device)
    same_out(x, ref.clip_tip_reads(None), ctx)
    return x


def test_gpu_tips_random_tiny_graphs(dg):
    n = n_changed = 0
    for seed in range(400):
        rng = np.random.default_rng(53000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14))) \
            if seed % 2 else error_reads(rng)
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = TipPolicyDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        dg.build(ids, off, k)
        ranks = [int(rng.integers(1, len(vocab) + 1))] if seed % 3 == 0 and len(vocab) else []
        min_length = int(rng.integers(1, k + 4))
        x = same_tips(dg, ref, min_length, ranks, "seed %d" % seed, on_device=seed % 3 == 1)
        n_changed += int(host(x)["changed"].any())
        flags = (rng.random(ref.sizes()["nodes"]) < 0.2).astype(np.uint8)
        try:
            ref.remove_nodes(flags)
        except TypeError:                                      # multi-edge: the device refuses it too
            continue
        dg.remove_nodes(flags)
        same_tips(dg, ref, min_length, ranks, "seed %d after remove_nodes" % seed)
        n += 1
    assert n >= 250 and n_changed >= 30, (n, n_changed)


@pytest.mark.parametrize("name", FIXTURES)
def test_gpu_tips_fixtures(dg, name):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input(name)
    for k in (1, 3, 5):
        try:
            ref = TipPolicyDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        dg.build(ids, off, k, ps, pe)
        same_tips(dg, ref, k + 1, (), "%s k=%d" % (name, k))
        same_tips(dg, ref, k + 1, (), "%s k=%d on device" % (name, k), on_device=True)


def test_gpu_host_flags_against_the_held_policy(dg):
    """host clip flags (the policy's, all ones, random) give what the loop gives for them; the held policy is dropped
    by host flags, and AMIRA_E_STATE follows"""
    from amira_b200 import _lib, synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 6000)
    ref = TipPolicyDevice().build(ids, off, 5)
    dg.build(ids, off, 5)
    _, clip = dg.tip_policy(6, want_clip=True)
    held = dg.clip_tip_reads(None)
    same_out(held, dg.clip_tip_reads(clip), "policy flags from the host")
    rng = np.random.default_rng(11)
    for flags in (np.ones_like(clip), (rng.random(len(clip)) < 0.5).astype(np.uint8)):
        same_out(dg.clip_tip_reads(flags), ref.clip_tip_reads(flags), "host flags")
    assert host(held)["changed"].sum() > 0
    with pytest.raises(_lib.AmiraLibraryError):
        dg.clip_tip_reads(None)                                # host flags overwrote the held ones


def test_gpu_tip_refusals(dg):
    from amira_b200 import _lib, synth
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 3000)
    dg.build(ids, off, 3)
    Q = dg.tip_count()
    assert Q > 0
    L, n = dg._lib, C.c_int64()
    assert L.amira_gmg_clip_tip_reads(dg._h, None, C.byref(n), *[None] * 6, 0) == _lib.E_STATE
    bad = np.zeros(Q, np.uint8)
    bad[Q // 2] = 2
    assert L.amira_gmg_clip_tip_reads(dg._h, bad.ctypes.data_as(C.c_void_p), C.byref(n), *[None] * 6, 0) == _lib.E_ARG
    with pytest.raises(ValueError):
        dg.clip_tip_reads(bad)
    with pytest.raises(ValueError):
        dg.clip_tip_reads(np.zeros(Q + 1, np.uint8))
    assert L.amira_gmg_tip_policy(dg._h, 4, None, 3, C.byref(n), None) == _lib.E_ARG
    dg.tip_policy(4)
    assert L.amira_gmg_clip_tip_reads(dg._h, None, C.byref(n), *[None] * 6, 0) == _lib.OK
    dg.filter_graph(2, 1)                                      # a new graph: the policy is gone
    if dg.tip_count():
        assert L.amira_gmg_clip_tip_reads(dg._h, None, C.byref(n), *[None] * 6, 0) == _lib.E_STATE


def test_gpu_a_junction_with_more_than_32_tips(dg):
    reads = {**{"t%d" % i: TRUE for i in range(60)}, **{"e%d" % i: TRUE[:-1] + ["+x%d" % i] for i in range(40)},
             **{"s%d" % i: ["-y%d" % i] + TRUE[1:] for i in range(36)}}
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    for k in (1, 3):
        ref = TipPolicyDevice().build(ids, off, k)
        dg.build(ids, off, k)
        x = host(same_tips(dg, ref, k + 1, (), "k=%d" % k))
        assert len(dg.tips()["tip_unitig"]) == 78 and x["changed"].sum() == 76 and x["tip_clipped"].sum() == 76


SCALE = [("c2", 20000, 3), ("c2", 20000, 5), ("c3", 60000, 3), ("c3", 60000, 5)]


@pytest.mark.parametrize("cfg_name,n_reads,k", SCALE)
def test_gpu_tips_synthetic(dg, cfg_name, n_reads, k):
    """unfiltered, after filter_graph(3, 1) and after filter_graph(1, 2), against the loops with spared ranks; then
    clip_compacted_tips on a lazy graph trimmed by remove_short_linear_paths(4) against the same on a host-edited graph,
    and the rebuild from the device CSR (with its call count) against the oracle's build of its host copy"""
    from amira_b200 import GeneMerGraph, encode, synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    ref = TipPolicyDevice().build(ids, off, k)
    for filt in (None, (3, 1), (1, 2)):
        ref.build(ids, off, k)
        dg.build(ids, off, k)
        if filt:
            for g in (dg, ref):
                g.filter_graph(*filt)
        x = same_tips(dg, ref, k + 1, (3, 7), (filt, "host outputs"))
        same_out(dg.clip_tip_reads(None, on_device=True), x, (filt, "device outputs"))
        assert filt or host(x)["changed"].sum() > 0
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS[cfg_name].vocab))
    enc = encode.EncodedReads(reads)
    lazy, hst = GeneMerGraph(enc, k), GeneMerGraph(enc, k)
    for g in (lazy, hst):
        g.remove_short_linear_paths(4)
    hst._touch()
    e = lazy.clip_compacted_tips(k + 1)
    assert lazy.__dict__["_lazy"] and e._device is not None
    e2 = hst.clip_compacted_tips(k + 1)
    same_out({f: getattr(e, f) for f in FIELDS}, {f: getattr(e2, f) for f in FIELDS}, "lazy against host-edited")
    assert e2.reads == e.reads
    g2 = GeneMerGraph(e, k)
    assert O.diff_arrays(g2._require_device_state().arrays(), TipPolicyDevice().build(e.ids, e.off, k).arrays()) == []


def test_gpu_rebuild_from_the_device_csr_with_its_call_count(dg):
    """the clipped device CSR rebuilt with n_calls on the handle is bit-exact against the oracle's build of the host
    copy, and holds fewer tips"""
    from amira_b200 import synth
    from amira_b200.device_graph import DeviceGraph
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 20000)
    dg.build(ids, off, 5)
    before = dg.tip_count()
    dg.tip_policy(6)
    x = dg.clip_tip_reads(None, on_device=True)
    h2 = DeviceGraph(0)
    h2.build(x["ids"], x["off"], 5, on_device=True, n_calls=len(x["ids"]))
    hx = host(x)
    want = TipPolicyDevice().build(hx["ids"], hx["off"], 5).arrays()
    assert O.diff_arrays(h2.arrays(), want) == []
    assert h2.tip_count() < before
    h2.close()


def test_gpu_tips_after_replayed_resident_builds(dg):
    import torch
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 8000)
    d_ids, d_off = torch.from_numpy(ids.copy()).cuda(), torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    ref = TipPolicyDevice().build(ids, off, 3)
    ref.tip_policy(4)
    want = ref.clip_tip_reads(None)
    for _ in range(3):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
        same_out(dg.tips(), ref.tips(), "replayed", TIP_FIELDS)
        dg.tip_policy(4)
        same_out(dg.clip_tip_reads(None), want, "replayed")
        same_out(dg.clip_tip_reads(None, on_device=True), want, "replayed, on device")


def test_gpu_tips_on_empty_graphs(dg):
    """an emptied graph and an empty read set: no tip, the output is the input"""
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input("synth_c2_2000")
    dg.build(ids, off, 3, ps, pe)
    dg.filter_graph(10**9, 1)
    assert dg.sizes()["nodes"] == 0 and dg.tip_count() == 0 and dg.tip_policy(4) == 0
    for clip in (None, np.zeros(0, np.uint8)):
        for on_device in (False, True):
            x = host(dg.clip_tip_reads(clip, on_device=on_device))
            assert np.array_equal(x["ids"], ids) and np.array_equal(x["off"], off) and not x["changed"].any()
            assert np.array_equal(x["pos_start"], ps) and np.array_equal(x["pos_end"], pe)
    dg.build(np.zeros(0, np.int32), np.zeros(1, np.int64), 3)
    assert dg.tip_count() == 0 and dg.tip_policy(4) == 0
    x = dg.clip_tip_reads(None)
    assert x["off"].tolist() == [0] and len(x["ids"]) == 0 and len(x["changed"]) == 0


def test_gpu_tip_calls_keep_caches_and_filter_masks(dg):
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    ref = TipPolicyDevice().build(ids, off, 3)
    dg.build(ids, off, 3)
    for g in (dg, ref):
        g.filter_graph(3, 1)
    nk, ek = dg.filter_masks()
    assert not nk.all()
    dg.tip_policy(4)
    dg.clip_tip_reads(None)                                    # the first calls reserve the buffers
    want = {"tips": dg.tips(), "bubbles": dg.bubbles(), "unitigs": dg.unitigs(), "paths": dg.read_unitig_paths()}
    n = dg.kernel_launches()
    same_tips(dg, ref, 4, (), on_device=True)
    m = dg.kernel_launches()
    for name, f in (("tips", dg.tips), ("bubbles", dg.bubbles), ("unitigs", dg.unitigs), ("paths", dg.read_unitig_paths)):
        x = f()
        assert all(np.array_equal(x[k], want[name][k]) for k in x), name
    assert dg.kernel_launches() == m and m > n
    x, y = dg.filter_masks()
    assert np.array_equal(x, nk) and np.array_equal(y, ek)


def test_gpu_tip_and_bubble_calls_interleaved(dg):
    """bubble_policy -> tips -> tip_policy -> clip_tip_reads -> correct_bubble_reads(None) succeeds and gives what
    bubble_policy -> correct_bubble_reads(None) gives; and the tip policy survives bubble calls in turn"""
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 20000)
    dg.build(ids, off, 5)
    dg.bubble_policy((5,))
    want = dg.correct_bubble_reads(None)
    dg.build(ids, off, 5)
    dg.bubble_policy((5,))
    dg.tips()
    dg.tip_policy(6, (5,))
    clip_want = dg.clip_tip_reads(None)
    same_out(dg.correct_bubble_reads(None), want, "bubbles after tips",
             ("ids", "off", "pos_start", "pos_end", "changed", "branch_rewritten"))
    dg.bubbles()
    dg.bubble_policy((5,))
    same_out(dg.clip_tip_reads(None), clip_want, "tips after bubbles")
    assert host(want, ("changed",))["changed"].sum() > 0 and host(clip_want)["changed"].sum() > 0


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def test_gpu_tip_calls_refuse_a_sharded_handle():
    n = _n_gpus()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    from tests.helpers import ROOT
    from tests.test_sharded import _free_port
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "sharded_tips_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0 and "SHARDED_TIPS OK" in res.stdout, (res.stdout[-3000:], res.stderr[-3000:])
