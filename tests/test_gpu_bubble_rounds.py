"""amira_gmg_bubble_policy and correct_bubbles_until_stable on the GPU: the policy kernel against replace_loop (its
definition as a plain loop) and against the numpy policy GeneMerGraph._bubble_winners, array-equal, on random tiny
graphs, the fixtures and synthetic inputs unfiltered and filtered, with random spared genes; exact ties and a bubble of
more than 32 branches; the correction with the device-held policy against the same call with the host replace_with;
correct_bubbles_until_stable against rounds_loop (tests/bubble_rounds_reference.py) and the final graph against the C
oracle's build of the final reads; six rounds of policy, correction and rebuild from the device CSR with the old
tensors dropped, bit-exact every round; no export on the handle during the rounds; AMIRA_E_STATE without a policy."""
import gc
from fractions import Fraction

import numpy as np
import pytest

from amira_b200 import _lib
from oracle import gmg_oracle as O
from tests.bubble_correction_reference import CorrectionDevice, replace_loop
from tests.bubble_rounds_reference import PolicyDevice, rounds_loop, spared_nodes
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
        assert np.array_equal(x[f].view(np.uint32) if f == "branch_rewritten" else x[f], y[f]), (ctx, f)


def check_policy(dg, ranks, u=None, ctx=""):
    """the device policy against replace_loop and _bubble_winners over the device's own (tested) unitigs and bubbles"""
    from amira_b200.construct_graph import GeneMerGraph
    bub, u = dg.bubbles(), u if u is not None else dg.unitigs()
    amr = np.asarray(dg.nodes_containing(ranks), bool) if len(ranks) else np.zeros(len(u["node_unitig"]), bool)
    n, rw = dg.bubble_policy(ranks, want_replace_with=True)
    want = replace_loop(u, bub, amr)
    assert np.array_equal(rw, want), ctx
    assert np.array_equal(rw, GeneMerGraph._bubble_winners(bub, u, amr)), ctx
    assert n == int((want >= 0).sum()) and dg.bubble_policy(ranks) == n, ctx
    return rw


def random_ranks(rng, n_genes):
    return [int(x) for x in rng.choice(np.arange(1, n_genes + 1), int(rng.integers(0, 3)), replace=False)] \
        if n_genes and rng.random() < 0.5 else []


def test_gpu_policy_random_tiny_graphs(dg):
    n = n_rep = 0
    for seed in range(400):
        rng = np.random.default_rng(54000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14))) \
            if seed % 2 else error_reads(rng)
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = PolicyDevice().build(ids, off, k)
        except AssertionError:                                 # palindromic window
            continue
        dg.build(ids, off, k)
        ranks = random_ranks(rng, len(vocab))
        a = ref.arrays()
        u = unitig_loop(a)
        rw = check_policy(dg, ranks, u, seed)
        assert np.array_equal(rw, ref.bubble_policy(ranks, True)[1]), seed
        assert np.array_equal(replace_loop(u, ref.bubbles(), spared_nodes(a, ranks)), rw), seed
        n_rep += int((rw >= 0).any())
        n += 1
    assert n >= 300 and n_rep >= 40, (n, n_rep)


@pytest.mark.parametrize("name", FIXTURES)
def test_gpu_policy_fixtures(dg, name):
    from tests.helpers import load_input
    vocab, ids, off, ps, pe = load_input(name)
    rng = np.random.default_rng(11)
    for k in (1, 3, 5):
        try:
            dg.build(ids, off, k, ps, pe)
        except AssertionError:
            continue
        check_policy(dg, [], ctx=(name, k))
        check_policy(dg, random_ranks(rng, len(vocab)) or [1], ctx=(name, k, "spared"))


SCALE = [("c2", 20000, 3), ("c2", 20000, 5), ("c3", 60000, 3), ("c3", 60000, 5)]


@pytest.mark.parametrize("cfg_name,n_reads,k", SCALE)
def test_gpu_policy_synthetic(dg, cfg_name, n_reads, k):
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    rng = np.random.default_rng(5)
    V = int(np.abs(ids).max())
    for filt in (None, (3, 1), (1, 2)):
        dg.build(ids, off, k)
        if filt:
            dg.filter_graph(*filt)
        rw = check_policy(dg, [], ctx=filt)
        assert filt or (rw >= 0).sum() > 0
        check_policy(dg, [int(x) for x in rng.choice(np.arange(1, V + 1), 20, replace=False)], ctx=(filt, "spared"))


def test_gpu_policy_ties_and_wide_bubbles(dg):
    """bubbles of up to 40 one-node and 6 two-node branches between s a and b t at k = 1, where a one-node branch's
    coverage is its read count: equal means and equal reads leave the index to decide, a two-node branch ties a
    one-node one on the mean, and the most reads decide between the branches of the highest mean"""
    def bubble(counts, two=(), half=()):
        """counts / two: the reads through each one-node / two-node branch; half: per two-node branch the reads
        "a y" plus "z b", which add 1 to the coverage of each of its nodes but run the branch only in part"""
        reads, r = {}, 0
        runs = [(c, ["+x%d" % i]) for i, c in enumerate(counts)] + [(c, ["+y%d" % i, "+z%d" % i]) for i, c in enumerate(two)]
        for c, mid in runs:
            for _ in range(c):
                reads["r%d" % r] = ["+s", "+a"] + mid + ["+b", "+t"]
                r += 1
        for i, c in enumerate(half):
            for _ in range(c):
                reads["r%d" % r], reads["r%d" % (r + 1)] = ["+a", "+y%d" % i], ["+z%d" % i, "+b"]
                r += 2
        vocab = O.build_vocabulary(reads)
        return O.encode_reads(reads, vocab)[:2]
    # (one-node reads, two-node reads, half reads, the branch kept): index only; index only; mean, then index; index only
    # over 33 branches; the reads break a tie of means; again over four branches; the mean wins over the index; the
    # reads win over the index
    for counts, two, half, want in (([2] * 40, (), (), 0), ([2] * 40, [2] * 6, (), 0),
                                    ([1] * 20 + [3] + [1] * 19, [3] * 6, (), 20), ([2] * 33, (), (), 0),
                                    ([3], [2], [1], 0), ([3, 3], [2, 2], [1, 1], 0), ([2, 1], [2], [1], 2),
                                    ((), [2, 3], [1, 0], 1)):
        ids, off = bubble(counts, two, half)
        dg.build(ids, off, 1)
        bub, u = dg.bubbles(), dg.unitigs()
        assert len(bub["source"]) == 1 and len(bub["branch_unitig"]) == len(counts) + len(two)
        rw = check_policy(dg, [])
        kept = np.flatnonzero(rw < 0)
        assert len(kept) == 1
        bu = bub["branch_unitig"].tolist()
        mean = [Fraction(int(u["cov_sum"][b]), int(u["unitig_off"][b + 1] - u["unitig_off"][b])) for b in bu]
        rd = bub["branch_reads"].astype(np.int64)
        top = np.flatnonzero([m == max(mean) for m in mean])
        best = top[rd[top] == rd[top].max()]
        assert kept[0] == best[0] == want, (counts, two, half)   # the highest mean, then the most reads, then the first
        ref = PolicyDevice().build(ids, off, 1)
        assert np.array_equal(ref.bubble_policy([], True)[1], rw)


def test_gpu_correction_with_the_device_policy(dg):
    """correct_bubble_reads(None) after bubble_policy against the same call with the policy's replace_with from the
    host, all six outputs, to the host and to the device"""
    from amira_b200 import synth
    from tests.helpers import load_input
    inputs = [load_input("synth_c2_2000")[1:], tuple(synth.generate(synth.CONFIGS["c3"], 0, 20000)) + (None, None)]
    for ids, off, ps, pe in inputs:
        for k, filt in ((3, None), (5, (1, 2))):
            dg.build(ids, off, k, ps, pe)
            if filt:
                dg.filter_graph(*filt)
            for on_device in (False, True):
                _, rw = dg.bubble_policy([1, 2], want_replace_with=True)
                x = dg.correct_bubble_reads(None, on_device=on_device)
                y = dg.correct_bubble_reads(rw, on_device=on_device)
                same_out(x, y, (k, filt, on_device))
                assert filt or host(x)["changed"].any()
                with pytest.raises(_lib.AmiraLibraryError, match="status 9"):
                    dg.correct_bubble_reads(None)          # the host replace_with replaced the policy's


def test_gpu_no_policy_is_a_state_error(dg):
    reads = {**{"t%d" % i: ["+a", "+b", "+c", "+d", "+e", "+f", "+g"] for i in range(5)},
             "e": ["+a", "+b", "+c", "+x", "+e", "+f", "+g"]}
    ids, off, _, _ = O.encode_reads(reads, O.build_vocabulary(reads))
    dg.build(ids, off, 3)
    with pytest.raises(_lib.AmiraLibraryError, match="status 9"):
        dg.correct_bubble_reads(None)
    assert dg.bubble_policy([]) == 1
    assert dg.correct_bubble_reads(None)["changed"].tolist() == [0] * 5 + [1]
    dg.remove_nodes(np.zeros(dg.sizes()["nodes"], np.uint8))
    with pytest.raises(_lib.AmiraLibraryError, match="status 9"):
        dg.correct_bubble_reads(None)                          # the graph changed since the policy
    dg.build(ids[:0], off[:1], 3)
    assert dg.bubble_policy([]) == 0 and dg.correct_bubble_reads(None)["off"].tolist() == [0]


ROUNDS = [("c2", 20000, 3, None, (), False), ("c2", 20000, 5, (3, 1), (1, 7), False), ("c3", 40000, 3, (1, 2), (), False),
          ("c3", 40000, 5, None, (3,), False), ("c3", 40000, 5, (3, 1), (), False), ("c2", 20000, 3, None, (1,), True),
          ("c3", 20000, 5, None, (), True)]


@pytest.mark.parametrize("cfg_name,n_reads,k,filt,genes,host_edited", ROUNDS)
def test_gpu_until_stable_against_the_composition(cfg_name, n_reads, k, filt, genes, host_edited):
    """host_edited: round 1 on the host implementation (numpy CSR and flags), the later rounds on the device"""
    from amira_b200 import GeneMerGraph, encode, synth
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    names = synth.vocabulary_names(synth.CONFIGS[cfg_name].vocab)
    reads = synth.to_read_dict(ids, off, names)
    genes = {names[i] for i in genes}
    g = GeneMerGraph(encode.EncodedReads(reads), k)
    if filt:
        g.filter_graph(*filt)
    if host_edited:
        g._touch()
    graph, out = g.correct_bubbles_until_stable(30, genes, filt)
    assert graph.__dict__["_lazy"] and (filt or out.rounds[0]["steps"] > 0)
    assert not host_edited or len(out.rounds) >= 2 and out.rounds[0]["steps"] > 0
    want_g, want_e, want_changed, want_rounds = rounds_loop(g, 30, genes, filt, fast=True)
    assert out.rounds == want_rounds
    assert out.reads == want_e.reads and np.array_equal(out.changed, want_changed)
    for f in ("ids", "off"):
        assert np.array_equal(getattr(out, f), getattr(want_e, f)), f
    assert np.array_equal(out.branch_rewritten, want_e.branch_rewritten)
    ref = CorrectionDevice().build(out.ids, out.off, k)
    if filt and ref.sizes()["nodes"]:
        ref.filter_graph(*filt)
    assert O.diff_arrays(graph._arrays(), ref.arrays()) == []
    assert O.diff_arrays(want_g._arrays(), ref.arrays()) == []


def test_gpu_six_rounds_bit_exact(dg):
    """policy, correction to the device and a rebuild from the device CSR, six times over C3 with the previous CSR
    dropped after each correction: torch hands out recycled addresses, and the resident build replays its captured
    graph when the sizes repeat; every correction and every rebuild is checked against the oracle"""
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 20000)
    ref = PolicyDevice().build(ids, off, 5)
    dg.build(ids, off, 5)
    csr = None
    for r in range(6):
        n = dg.bubble_policy([])
        assert n == ref.bubble_policy([]), r
        x = dg.correct_bubble_reads(None, on_device=True)
        want = ref.correct_bubble_reads(None)
        same_out(x, want, r)
        del csr
        gc.collect()
        csr = x
        # the count the loop passes, or the one the build caches by address (even rounds), which recycled
        # addresses make stale: both must give the oracle's graph
        dg.build(x["ids"], x["off"], 5, on_device=True, n_calls=len(x["ids"]) if r % 2 else None)
        ref.build(want["ids"], want["off"], 5)
        assert O.diff_arrays(dg.arrays(), ref.arrays()) == [], r


def test_gpu_rounds_export_nothing(monkeypatch):
    """correct_bubbles_until_stable on a lazy graph calls no export on the handle, and both graphs stay lazy"""
    from amira_b200 import GeneMerGraph, encode, synth
    from amira_b200.device_graph import DeviceGraph
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 20000)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS["c3"].vocab))
    g = GeneMerGraph(encode.EncodedReads(reads), 5)
    calls = []
    for name in ("arrays", "unitigs", "bubbles", "read_unitig_paths", "nodes_containing", "arrays_reads_only"):
        def spy(self, *a, _f=getattr(DeviceGraph, name), _n=name, **kw):
            calls.append(_n)
            return _f(self, *a, **kw)
        monkeypatch.setattr(DeviceGraph, name, spy)
    graph, out = g.correct_bubbles_until_stable(30, {"g1"}, (1, 1))
    assert calls == [] and len(out.rounds) >= 2
    assert graph.__dict__["_lazy"] and g.__dict__["_lazy"]
