"""amira_gmg_gene_paths on the GPU against the loops of tests/gene_path_reference.py and the numpy implementation,
array by array: random tiny graphs before and after removals; the fixtures; 20 000-read subsamples of C2, C3 and C5
with the generator's AMR genes plus random genes, unfiltered, filtered and after clean_until_stable; the degenerate
key hash; the cache (no launch for the same ranks, recomputed for new ranks and after a filter, the other caches and
held policies kept); a cluster with more than 70 000 members; a node in more than 1 000 keys; bad ranks; replayed
resident builds; an empty graph; the sharded refusal."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from amira_b200.construct_graph import GeneMerGraph
from oracle import gmg_oracle as O
from tests.fake_device import OracleBackedDevice
from tests.gene_path_reference import gene_path_loop, marked_nodes, same_gene_paths
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dg():
    from amira_b200.device_graph import DeviceGraph
    g = DeviceGraph(0)
    yield g
    g.close()


def check(dg, a, ranks, ctx, loop=True):
    """the device against the numpy implementation over the oracle's arrays a (and the loops when `loop`)"""
    x = dg.gene_paths(ranks)
    marked = marked_nodes(a, ranks)
    want = GeneMerGraph._gene_paths_over(a, marked)
    same_gene_paths(x, want, ctx)
    if loop:
        same_gene_paths(want, gene_path_loop(a, marked), ctx)
    return x


def test_gpu_gene_paths_random_tiny_graphs(dg):
    n = n_clusters = 0
    for seed in range(300):
        rng = np.random.default_rng(81000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 30)), int(rng.integers(2, 9)), int(rng.integers(1, 16)))
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = OracleBackedDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        dg.build(ids, off, k)
        ranks = sorted(set(rng.integers(1, len(vocab) + 1, int(rng.integers(1, 4))).tolist())) if len(vocab) else []
        x = check(dg, ref.arrays(), ranks, "seed %d" % seed)
        n_clusters += len(x["n_complete"])
        flags = (rng.random(ref.sizes()["nodes"]) < 0.2).astype(np.uint8)
        try:
            ref.remove_nodes(flags)
        except TypeError:                                      # multi-edge: the device refuses it too
            continue
        dg.remove_nodes(flags)
        check(dg, ref.arrays(), ranks, "seed %d after remove_nodes" % seed)
        n += 1
    assert n >= 150 and n_clusters >= 200, (n, n_clusters)


@pytest.mark.parametrize("name", FIXTURES)
def test_gpu_gene_paths_fixtures(dg, name):
    from tests.helpers import load_input
    vocab, ids, off, ps, pe = load_input(name)
    rng = np.random.default_rng(len(name))
    for k in (1, 3, 5):
        try:
            ref = OracleBackedDevice().build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        dg.build(ids, off, k, ps, pe)
        for ranks in ([1], sorted(set(rng.integers(1, len(vocab) + 1, 6).tolist()))):
            check(dg, ref.arrays(), ranks, "%s k=%d" % (name, k))


def synth_ranks(cfg, rng, n_random=20):
    from amira_b200 import synth
    amr = synth._pool(cfg).amr.tolist()
    return sorted(set(amr + rng.integers(1, cfg.vocab + 1, n_random).tolist()))


SCALE = [("c2", 3), ("c3", 3), ("c3", 5), ("c5", 5)]


@pytest.mark.parametrize("cfg_name,k", SCALE)
def test_gpu_gene_paths_synthetic(dg, cfg_name, k):
    """20 000 reads: unfiltered and after filter_graph(3, 1) against the numpy implementation on the oracle's arrays;
    after clean_until_stable(6) a lazy graph against the same graph edited on the host; the AMR genes make clusters"""
    from amira_b200 import encode, synth
    cfg = synth.CONFIGS[cfg_name]
    ids, off = synth.generate(cfg, 0, 20000)
    rng = np.random.default_rng(5)
    ranks = synth_ranks(cfg, rng)
    amr = synth._pool(cfg).amr.tolist()
    ref = OracleBackedDevice()
    for filt in (None, (3, 1)):
        ref.build(ids, off, k)
        dg.build(ids, off, k)
        if filt:
            for g in (dg, ref):
                g.filter_graph(*filt)
        a = ref.arrays()
        for r in (ranks, amr[:1]):
            x = check(dg, a, r, (cfg_name, k, filt, len(r)), loop=False)
        assert filt or (x["n_complete"] > 0).sum() >= 2
    names = synth.vocabulary_names(cfg.vocab)
    genes = [names[r - 1] for r in amr]                                # few genes: the host path scans every node per gene
    enc = encode.EncodedReads(synth.to_read_dict(ids, off, names))
    lazy, _ = GeneMerGraph(enc, k).clean_until_stable(6)
    x = lazy.gene_paths(genes)
    assert lazy.__dict__["_lazy"]
    a = lazy._require_device_state().arrays()
    marked = marked_nodes(a, lazy._gene_ranks(genes))                  # ranks in the reads' own vocabulary
    same_gene_paths(x, GeneMerGraph._gene_paths_over(a, marked), "after clean_until_stable")
    lazy._touch()
    same_gene_paths(lazy.gene_paths(genes), x, "host-edited after clean_until_stable")


def test_gpu_gene_paths_degenerate_hash(dg):
    from amira_b200 import synth
    cfg = synth.CONFIGS["c3"]
    ids, off = synth.generate(cfg, 0, 20000)
    ranks = synth_ranks(cfg, np.random.default_rng(9), 200)
    dg.build(ids, off, 3)
    want = dg.gene_paths(ranks)
    assert len(want["n_complete"]) > 100
    try:
        dg.debug_layout(32)
        same_gene_paths(dg.gene_paths(ranks), want, "3-bit hash")
        dg.build(ids, off, 3)
        same_gene_paths(dg.gene_paths(ranks), want, "3-bit hash, rebuilt")
    finally:
        dg.debug_layout(0)
    same_gene_paths(dg.gene_paths(ranks), want, "full hash again")


def test_gpu_gene_paths_cache(dg):
    """the same ranks launch nothing; new ranks and a filter recompute; the unitig, bubble and tip caches, both held
    policies and the filter masks survive"""
    from amira_b200 import _lib, synth
    cfg = synth.CONFIGS["c3"]
    ids, off = synth.generate(cfg, 0, 6000)
    ranks = synth_ranks(cfg, np.random.default_rng(2))
    ref = OracleBackedDevice().build(ids, off, 3)
    dg.build(ids, off, 3)
    for g in (dg, ref):
        g.filter_graph(2, 1)
    nk, ek = dg.filter_masks()
    dg.bubble_policy(())
    dg.tip_policy(4)
    want = {"unitigs": dg.unitigs(), "bubbles": dg.bubbles(), "tips": dg.tips(), "paths": dg.read_unitig_paths(),
            "correct": dg.correct_bubble_reads(None), "clip": dg.clip_tip_reads(None)}
    x = check(dg, ref.arrays(), ranks, "first", loop=False)
    n = dg.kernel_launches()
    same_gene_paths(dg.gene_paths(ranks), x, "cached")
    assert dg.kernel_launches() == n
    check(dg, ref.arrays(), ranks[:3], "new ranks", loop=False)
    assert dg.kernel_launches() > n
    m = dg.kernel_launches()
    for name, f in (("unitigs", dg.unitigs), ("bubbles", dg.bubbles), ("tips", dg.tips), ("paths", dg.read_unitig_paths)):
        y = f()
        assert all(np.array_equal(y[k], want[name][k]) for k in y), name
    assert dg.kernel_launches() == m
    for name, y in (("correct", dg.correct_bubble_reads(None)), ("clip", dg.clip_tip_reads(None))):
        assert all(np.array_equal(y[k], want[name][k]) for k in y if y[k] is not None), name
    p, q = dg.filter_masks()
    assert np.array_equal(p, nk) and np.array_equal(q, ek)
    for g in (dg, ref):
        g.filter_graph(3, 1)
    m = dg.kernel_launches()
    check(dg, ref.arrays(), ranks[:3], "after a filter", loop=False)
    assert dg.kernel_launches() > m
    L, cnt = dg._lib, C.c_int64()
    assert L.amira_gmg_gene_paths(dg._h, None, 2, C.byref(cnt), *[None] * 14) == _lib.E_ARG
    assert L.amira_gmg_gene_paths(dg._h, None, -1, C.byref(cnt), *[None] * 14) == _lib.E_ARG


def test_gpu_a_cluster_with_more_than_70000_members(dg):
    """one context read 75 000 times (both orientations): one cluster, its members sorted by the CTA path of the
    segmented sort; and one gene in 1 200 contexts, whose node lies in every key"""
    ctx = ["+x1", "+x2", "+x3", "+amr", "+y1", "+y2", "+y3"]
    rc = [("-" if g[0] == "+" else "+") + g[1:] for g in ctx[::-1]]
    reads = {"r%d" % i: (ctx if i % 3 else rc) for i in range(75000)}
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    dg.build(ids, off, 3)
    a = dg.arrays()
    ranks = [vocab.index("amr") + 1]
    x = dg.gene_paths(ranks)
    same_gene_paths(x, GeneMerGraph._gene_paths_over(a, marked_nodes(a, ranks)), "75 000 members")
    assert len(x["n_complete"]) == 1 and x["members"].tolist() == list(range(75000))
    many = {}
    for i in range(1200):
        ctx = ["+e%d" % i, "+l%d" % i, "+amr", "+m", "+r%d" % i]   # +amr +m: one node shared by every context
        many["c%d" % i] = ctx
        many["p%d" % i] = ctx[2:4]
    vocab = O.build_vocabulary(many)
    ids, off, _, _ = O.encode_reads(many, vocab)
    ref = OracleBackedDevice().build(ids, off, 2)
    dg.build(ids, off, 2)
    ranks = [vocab.index("amr") + 1]
    x = check(dg, ref.arrays(), ranks, "a node in 1 200 keys", loop=False)
    assert len(x["n_complete"]) == 1200 and (x["occ_cluster"][x["occ_flanks"] != 3] == -2).all()


def test_gpu_gene_paths_after_replayed_resident_builds(dg):
    import torch
    from amira_b200 import synth
    cfg = synth.CONFIGS["c2"]
    ids, off = synth.generate(cfg, 0, 8000)
    d_ids, d_off = torch.from_numpy(ids.copy()).cuda(), torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    ranks = synth_ranks(cfg, np.random.default_rng(4))
    a = OracleBackedDevice().build(ids, off, 3).arrays()
    want = GeneMerGraph._gene_paths_over(a, marked_nodes(a, ranks))
    for _ in range(3):
        dg.build(d_ids, d_off, 3, on_device=True, wait=False)
        same_gene_paths(dg.gene_paths(ranks), want, "replayed")


def test_gpu_gene_paths_on_empty_graphs(dg):
    from tests.helpers import load_input
    _, ids, off, ps, pe = load_input("synth_c2_2000")
    dg.build(ids, off, 3, ps, pe)
    dg.filter_graph(10**9, 1)
    x = dg.gene_paths([1, 2, 3])
    assert all(len(x[f]) == 0 for f in ("occ_read", "key_state", "members")) and x["key_off"].tolist() == [0]
    dg.build(np.zeros(0, np.int32), np.zeros(1, np.int64), 3)
    x = dg.gene_paths([1])
    assert len(x["occ_read"]) == 0 and x["member_off"].tolist() == [0]


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def test_gpu_gene_paths_refuse_a_sharded_handle():
    n = _n_gpus()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    from tests.helpers import ROOT
    from tests.test_sharded import _free_port
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "sharded_gene_paths_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0 and "SHARDED_GENE_PATHS OK" in res.stdout, (res.stdout[-3000:], res.stderr[-3000:])
