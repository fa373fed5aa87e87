"""The references the GPU post-build tests compare with, checked against each other without a GPU:

* the C oracle's remove_nodes (one pass: multi-edge check, then removal) against the Python oracle's upstream-style
  remove_node one node at a time, on random tiny graphs where multi-edges, self edges and hairpins are common;
* the test double's numpy scans (linear_steps, junk_read_mask) against plain loops over the oracle's arrays;
* the test double's remove_nodes_without_reads_of and filter masks against the Python oracle."""
import numpy as np
import pytest

from oracle import c_oracle
from oracle import gmg_oracle as O
from tests.fake_device import OracleBackedDevice
from tests.test_random_small_cpu import random_reads

SEEDS = range(300)
ERROR_RATES = (0.0, 0.2, 0.5, 0.7, 0.75, 0.9, 1.0)


def tiny_case(seed):
    """-> (rng, reads, vocabulary, k, ids, off), or None for a palindromic window (the build raises)"""
    rng = np.random.default_rng(5000 + seed)
    reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
    k = int(rng.integers(1, 6))
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    try:
        O.OracleGraph(reads, k)
    except AssertionError:
        return None
    return rng, reads, vocab, k, ids, off


def random_flags(rng, n):
    return (rng.random(n) < rng.choice([0.0, 0.1, 0.5, 1.0])).astype(np.uint8)


# ---- loop restatements of upstream's per-node / per-read code, the references for the numpy versions ----
def linear_steps_loop(a):
    n = len(a["node_cov"])
    deg = (np.diff(a["fw_off"]) + np.diff(a["bw_off"])).astype(np.uint32)
    out = {"degree": deg}
    for side, off, edges in (("fw", a["fw_off"], a["fw_edges"]), ("bw", a["bw_off"], a["bw_edges"])):
        nxt, dr, ext = np.full(n, -1, np.int32), np.zeros(n, np.int8), np.zeros(n, np.uint8)
        for i in range(n):
            cnt = off[i + 1] - off[i]
            if (cnt == 1) if side == "fw" else (cnt > 0):
                e = edges[off[i]]
                t = a["edge_tgt"][e]
                nxt[i], dr[i] = t, a["edge_td"][e]
                ext[i] = deg[t] in (1, 2) and t != i
        out[side + "_next"], out[side + "_dir"], out[side + "_ext"] = nxt, dr, ext
    return out


def junk_read_mask_loop(a, error_rate):
    R = len(a["is_short"])
    out = np.zeros(R, np.uint8)
    for r in range(R):
        if a["is_short"][r]:
            out[r] = 2
            continue
        w = a["win_node"][a["win_off"][r]:a["win_off"][r + 1]].tolist()
        out[r] = w.count(-1) <= round(len(w) * (1 - error_rate))
    return out


ROUNDING_TIES = [(1, 0.5, 0), (3, 0.5, 2), (5, 0.5, 2), (5, 0.9, 0), (5, 0.7, 2), (2, 0.75, 0)]


def rounding_tie_reads(n):
    """k = 1 reads; after filter_graph(2, 1) read r (r = 0..n) has n windows of which exactly r are None (its first
    r genes are on no other read), read n + 1 has none and read n + 2 is empty (short) -> (ids, off)"""
    reads = [[1000 * (r + 1) + j for j in range(r)] + [j + 1 for j in range(r, n)] for r in range(n + 1)]
    reads.append([j + 1 for j in range(n)])
    reads.append([])
    off = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.int64)
    ids = np.concatenate([np.asarray(r, np.int32).reshape(-1) for r in reads])
    return ids, off


def rounding_tie_mask(n, rounded):
    """junk_read_mask of rounding_tie_reads(n) when round(n * (1 - error_rate)) == rounded"""
    return [int(r <= rounded) for r in range(n + 1)] + [1, 2]


def test_c_remove_nodes_matches_one_at_a_time_remove_node():
    n_cases = n_multi = n_removed = 0
    for seed in SEEDS:
        case = tiny_case(seed)
        if case is None:
            continue
        rng, reads, vocab, k, ids, off = case
        py, c = O.OracleGraph(reads, k), c_oracle.COracleGraph(ids, off, k)
        n_cases += 1
        if rng.random() < 0.4:                  # sometimes after a filter (the C oracle's edge map is rebuilt)
            py.filter_graph(2, 1)
            c.filter_graph(2, 1)
        for step in range(3):
            before = c.arrays()
            assert O.diff_arrays(py.arrays(vocab), before) == [], (seed, step)
            flags = random_flags(rng, len(before["node_cov"]))
            errs = []
            for g, arg in ((py, np.flatnonzero(flags).tolist()), (c, flags)):
                try:
                    g.remove_nodes(arg)
                    errs.append(None)
                except TypeError:
                    errs.append(TypeError)
            assert errs[0] == errs[1], (seed, step, errs)
            if errs[0] is TypeError:
                n_multi += 1
                assert O.diff_arrays(before, c.arrays()) == [], (seed, step, "C oracle changed on TypeError")
                assert O.diff_arrays(before, py.arrays(vocab)) == [], (seed, step, "Python oracle changed on TypeError")
                break
            n_removed += int(flags.sum())
            assert O.diff_arrays(py.arrays(vocab), c.arrays()) == [], (seed, step)
    assert n_cases > 200 and n_multi > 10 and n_removed > 500, (n_cases, n_multi, n_removed)


def test_c_oracle_removals_after_a_filter_on_a_large_graph():
    """the multi-edge check rebuilds the edge map a filter dropped, for more edges than its initial size"""
    from amira_b200 import synth
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 3000)
    fresh, c = c_oracle.COracleGraph(ids, off, 3), c_oracle.COracleGraph(ids, off, 3)
    c.filter_graph(1, 1)                                    # removes nothing, drops the map
    assert len(c.arrays()["edge_cov"]) > 4096 * 4
    fresh.remove_low_coverage_components(5)
    c.remove_low_coverage_components(5)
    assert O.diff_arrays(fresh.arrays(), c.arrays()) == []
    c.filter_graph(2, 1)
    flags = np.zeros(len(c.arrays()["node_cov"]), np.uint8)
    flags[::3] = 1
    c.remove_nodes(flags)
    k1 = c_oracle.COracleGraph(ids, off, 1)
    k1.filter_graph(2, 1)
    with pytest.raises(TypeError):
        k1.remove_nodes(np.ones(len(k1.arrays()["node_cov"]), np.uint8))


def test_remove_nodes_rejects_wrong_flag_count():
    c = c_oracle.COracleGraph(np.array([1, 2, 3, 4], np.int32), np.array([0, 4], np.int64), 3)
    with pytest.raises(AssertionError):
        c.remove_nodes(np.zeros(3, np.uint8))


def test_double_scans_equal_loop_versions():
    """numpy linear_steps / junk_read_mask of the test double == the loops, on graphs with None windows"""
    n_none = 0
    for seed in SEEDS:
        case = tiny_case(seed)
        if case is None:
            continue
        rng, reads, vocab, k, ids, off = case
        d = OracleBackedDevice().build(ids, off, k)
        for op in range(2):
            a = d.arrays()
            n_none += int((a["win_node"] < 0).sum())
            got, want = d.linear_steps(), linear_steps_loop(a)
            assert got.keys() == want.keys()
            for f in want:
                assert got[f].dtype == want[f].dtype and np.array_equal(got[f], want[f]), (seed, op, f)
            for er in ERROR_RATES:
                assert np.array_equal(d.junk_read_mask(er), junk_read_mask_loop(a, er)), (seed, op, er)
            try:
                if op == 0:
                    d.filter_graph(int(rng.integers(1, 4)), int(rng.integers(1, 3)))
                else:
                    d.remove_nodes(random_flags(rng, d.sizes()["nodes"]))
            except TypeError:
                break
    assert n_none > 1000, n_none


@pytest.mark.parametrize("n,error_rate,want", ROUNDING_TIES)
def test_junk_read_mask_rounds_half_to_even(n, error_rate, want):
    """reads of n windows with 0..n of them None: kept iff #None <= round(n * (1 - er)); the products land on or
    next to .5 (5 * (1 - 0.9) = 0.4999999999999999, 5 * (1 - 0.7) = 1.5000000000000002)"""
    assert round(n * (1 - error_rate)) == want
    ids, off = rounding_tie_reads(n)
    d = OracleBackedDevice().build(ids, off, 1)
    d.filter_graph(2, 1)
    a = d.arrays()
    assert [int((a["win_node"][a["win_off"][r]:a["win_off"][r + 1]] < 0).sum()) for r in range(n + 1)] == list(range(n + 1))
    mask = d.junk_read_mask(error_rate)
    assert mask.tolist() == rounding_tie_mask(n, want)
    assert np.array_equal(mask, junk_read_mask_loop(a, error_rate))


def test_double_remove_nodes_without_reads_of_matches_python_oracle():
    """remove_non_AMR_associated_nodes on the Python oracle's records: the reads of the nodes holding a gene, and
    every node on none of them removed with remove_node; the double's keep flags name exactly the removed objects"""
    n_partial = 0
    for seed in SEEDS:
        case = tiny_case(seed)
        if case is None:
            continue
        rng, reads, vocab, k, ids, off = case
        py = O.OracleGraph(reads, k)
        d = OracleBackedDevice().build(ids, off, k)
        ranks = rng.integers(0, len(vocab) + 2, int(rng.integers(0, 4))).tolist()
        genes = {vocab[r - 1] for r in ranks if 1 <= r <= len(vocab)}
        nodes = list(py.nodes.values())
        wanted = set()
        for n in nodes:
            if genes.intersection(name for name, _ in n.names):
                wanted.update(n.reads)
        doomed = [i for i, n in enumerate(nodes) if not wanted.intersection(n.reads)]
        before = d.arrays()
        errs = []
        for op in (lambda: py.remove_nodes(doomed), lambda: d.remove_nodes_without_reads_of(ranks)):
            try:
                op()
                errs.append(None)
            except TypeError:
                errs.append(TypeError)
        assert errs[0] == errs[1], (seed, errs)
        if errs[0] is TypeError:
            with pytest.raises(RuntimeError):
                d.filter_masks()
            continue
        assert O.diff_arrays(py.arrays(vocab), d.arrays()) == [], seed
        nk, ek = d.filter_masks()
        want_nk = np.ones(len(nodes), bool)
        want_nk[doomed] = False
        assert np.array_equal(nk, want_nk), seed
        assert np.array_equal(ek, want_nk[before["edge_src"]] & want_nk[before["edge_tgt"]]), seed
        n_partial += 0 < len(doomed) < len(nodes)
    assert n_partial > 30, n_partial


def test_double_filter_masks_follow_the_last_call():
    ids = np.array([1, 2, 3, 4, 1, 2, 3, 5, 7, 8, 9], np.int32)
    d = OracleBackedDevice().build(ids, np.array([0, 4, 8, 11], np.int64), 3)
    with pytest.raises(RuntimeError):
        d.filter_masks()
    d.filter_graph(2, 1)
    nk, ek = d.filter_masks()
    assert nk.tolist() == [True, False, False, False] and len(ek) == 4 and not ek.any()
    d.linear_steps()                          # the library reuses the masks' buffer: they are gone
    with pytest.raises(RuntimeError):
        d.filter_masks()
    d.remove_nodes(np.ones(1, np.uint8))
    nk, ek = d.filter_masks()
    assert nk.tolist() == [False] and len(ek) == 0
    d.remove_nodes(np.zeros(0, np.uint8))     # empty graph: masks of zero nodes
    assert [len(m) for m in d.filter_masks()] == [0, 0]
