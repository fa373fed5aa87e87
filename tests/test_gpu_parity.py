"""GPU parity through the C ABI: amira_gmg_build / filter / exports vs the golden vectors from the
unmodified upstream class and vs the C oracle on seeded synthetic inputs (bit-exact, all fields)."""
import numpy as np
import pytest

from tests.helpers import EXPECTED, GOLDEN_KEYS, STAGE_ORDER, apply_stage, load_input

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dg():
    from amira_b200.device_graph import DeviceGraph
    g = DeviceGraph(0)
    yield g
    g.close()


@pytest.mark.parametrize("key", GOLDEN_KEYS)
def test_gpu_matches_upstream_golden(dg, key):
    from oracle import gmg_oracle as O
    exp = EXPECTED[key]
    vocab, ids, off, ps, pe = load_input(exp["input"])
    dg.build(ids, off, exp["k"], ps, pe)
    for stage in STAGE_ORDER:
        want = exp["stages"].get(stage)
        if want is None:
            break
        if "raises" in want:
            with pytest.raises(TypeError):
                apply_stage(dg, stage)
            break
        apply_stage(dg, stage)
        a = dg.arrays()
        assert O.summary(a) == want["summary"], (key, stage)
        got = O.digest_arrays(a)
        assert got == want["digest"], (key, stage, [f for f in got if got[f] != want["digest"][f]])


SYNTH = [("c2", 20000, 3, False), ("c2", 20000, 5, True), ("c3", 60000, 3, False), ("c3", 60000, 7, False),
         ("c4", 50000, 3, False), ("c5", 40000, 5, False), ("c5", 5000, 15, False), ("c3", 3000, 1, False)]


@pytest.mark.parametrize("cfg_name,n_reads,k,with_pos", SYNTH)
def test_gpu_matches_c_oracle_on_synthetic(dg, cfg_name, n_reads, k, with_pos):
    from amira_b200 import synth
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    cfg = synth.CONFIGS[cfg_name]
    ids, off = synth.generate(cfg, 0, n_reads)
    ps = pe = None
    if with_pos:
        ps, pe = synth.positions_for(off, 7)
    ref = c_oracle.COracleGraph(ids, off, k, ps, pe)
    dg.build(ids, off, k, ps, pe)
    assert O.diff_arrays(dg.arrays(), ref.arrays()) == []
    if k == 1:
        return
    ref.remove_low_coverage_components(5)
    dg.remove_low_coverage_components(5)
    assert O.diff_arrays(dg.arrays(), ref.arrays()) == []
    ref.filter_graph(3, 1)
    dg.filter_graph(3, 1)
    assert O.diff_arrays(dg.arrays(), ref.arrays()) == []
    ref.filter_graph(4, 6)
    dg.filter_graph(4, 6)
    assert O.diff_arrays(dg.arrays(), ref.arrays()) == []


@pytest.mark.parametrize("mask", [1, 2, 3, 5, 7, 8, 16, 24])
@pytest.mark.parametrize("cfg_name,n_reads,k", [("c3", 30000, 3), ("c5", 20000, 5), ("c4", 20000, 7)])
def test_gpu_every_table_layout(dg, mask, cfg_name, n_reads, k):
    """32-byte node slots (packed and unpacked keys) and 32-byte edge slots give the same graph as the 16-byte ones"""
    from amira_b200 import synth
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    ids, off = synth.generate(synth.CONFIGS[cfg_name], 0, n_reads)
    ref = c_oracle.COracleGraph(ids, off, k)
    dg.debug_layout(mask)
    try:
        dg.build(ids, off, k)
        assert O.diff_arrays(dg.arrays(), ref.arrays()) == []
        ref.remove_low_coverage_components(5)
        dg.remove_low_coverage_components(5)
        ref.filter_graph(3, 1)
        dg.filter_graph(3, 1)
        assert O.diff_arrays(dg.arrays(), ref.arrays()) == []
    finally:
        dg.debug_layout(0)


def test_gpu_id_width_is_remeasured(dg):
    """a handle that has only seen small gene ids must notice larger ones (packed keys are sized from the largest |id|)"""
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    rng = np.random.default_rng(5)
    off = np.arange(0, 3001, 30).astype(np.int64)
    for vmax in (20, 5000, 2_000_000, 900_000_000, 50):
        ids = (rng.integers(1, vmax + 1, off[-1]) * rng.choice([-1, 1], off[-1])).astype(np.int32)
        ids[:40] = np.tile(ids[:5], 8)           # some repeats so that nodes get coverage > 1
        for k in (3, 5):
            dg.build(ids, off, k)
            assert O.diff_arrays(dg.arrays(), c_oracle.COracleGraph(ids, off, k).arrays()) == [], (vmax, k)


def test_gpu_edge_cases(dg):
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    # no reads at all, any k (upstream tests/test_gene_mer_graph.py:14-36)
    for k in (0, 3):
        dg.build(np.zeros(0, np.int32), np.zeros(1, np.int64), k)
        assert O.summary(dg.arrays())["nodes"] == 0
    # only empty / short reads
    off = np.array([0, 0, 2, 2, 4, 4], np.int64)
    ids = np.array([1, 2, -2, -1], np.int32)
    dg.build(ids, off, 3)
    a = dg.arrays()
    assert a["is_short"].tolist() == [1, 1, 1, 1, 1] and len(a["node_cov"]) == 0
    # ragged: empty reads between real ones, reads longer than a tile, a tile boundary inside a read
    rng = np.random.default_rng(1)
    lens = np.concatenate([[0, 0, 3000, 0, 1, 2, 3, 0, 1500], rng.integers(0, 40, 500), [0, 0]])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    ids = (rng.integers(1, 50, off[-1]) * rng.choice([-1, 1], off[-1])).astype(np.int32)
    for k in (1, 3, 5):
        ref = c_oracle.COracleGraph(ids, off, k)
        dg.build(ids, off, k)
        assert O.diff_arrays(dg.arrays(), ref.arrays()) == [], k
    # palindromic even-k window -> AssertionError like upstream (construct_gene_mer.py:23-25)
    with pytest.raises(AssertionError):
        dg.build(np.array([5, -5, 7], np.int32), np.array([0, 3], np.int64), 2)
    with pytest.raises(AssertionError):
        dg.build(np.array([5, 6, 7], np.int32), np.array([0, 3], np.int64), 0)
    # the handle survives an error
    dg.build(np.array([5, 6, 7, 8], np.int32), np.array([0, 4], np.int64), 3)
    assert dg.sizes()["nodes"] == 2


def test_gpu_device_resident_input(dg):
    import torch
    from amira_b200 import synth
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 10000)
    d_ids = torch.from_numpy(ids).cuda()
    d_off = torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    dg.build(d_ids, d_off, 3, on_device=True)
    assert O.diff_arrays(dg.arrays(), c_oracle.COracleGraph(ids, off, 3).arrays()) == []


def test_gpu_python_class_matches_upstream_snapshots(golden_small):
    """the drop-in GeneMerGraph class on the real device: node / edge SHA keys, insertion orders, coverages,
    per-read lists, short reads, filters -- against full dumps of the unmodified upstream class"""
    from amira_b200 import GeneMerGraph
    from tests.graph_snapshot import check_small_cases
    check_small_cases(GeneMerGraph, golden_small, pytest)


def test_gpu_python_class_on_a_fixture_scale_input():
    """the class, through encode -> C ABI -> materialisation, agrees with the array-level build it wraps"""
    from amira_b200 import GeneMerGraph, synth
    from oracle import c_oracle
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 3000)
    names = synth.vocabulary_names(synth.CONFIGS["c2"].vocab)
    reads = synth.to_read_dict(ids, off, names)
    g = GeneMerGraph(reads, 3)
    ref = c_oracle.COracleGraph(ids, off, 3).arrays()
    assert len(g.get_nodes()) == len(ref["node_cov"]) and len(g.get_edges()) == len(ref["edge_cov"])
    assert [n.get_node_coverage() for n in g.all_nodes()] == ref["node_cov"].tolist()
    assert [e.get_edge_coverage() for e in g.get_edges().values()] == ref["edge_cov"].tolist()
    assert [n.get_component() for n in g.all_nodes()] == ref["node_comp"].tolist()
    rid = list(reads)
    assert [len(g.get_readNodes().get(r, [])) for r in rid] == np.diff(ref["win_off"]).tolist()
    g.remove_low_coverage_components(5)
    g.filter_graph(3, 1)
    r2 = c_oracle.COracleGraph(ids, off, 3)
    r2.remove_low_coverage_components(5)
    r2.filter_graph(3, 1)
    a2 = r2.arrays()
    assert [n.get_node_coverage() for n in g.all_nodes()] == a2["node_cov"].tolist()
    assert len(g.get_edges()) == len(a2["edge_cov"])
    assert sorted(g.get_reads_to_correct()) == sorted(rid[i] for i in np.flatnonzero(a2["to_correct"]).tolist())


def test_gpu_streamed_host_input(dg):
    """host input large enough to arrive in pieces (one insert launch per piece) gives the oracle's graph"""
    from amira_b200 import synth
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    ids, off = synth.generate(synth.CONFIGS["c5"], 0, 160000)
    assert len(ids) >= 4 * (1 << 20)
    for k in (5, 3):
        dg.build(ids, off, k)
        assert O.diff_arrays(dg.arrays(), c_oracle.COracleGraph(ids, off, k).arrays()) == [], k


def test_gpu_key_width_follows_the_data_down_again():
    """after an input with huge gene ids the handle goes back to the compact layout for small ids (timing aside,
    the graphs must stay exact across the switches)"""
    from amira_b200.device_graph import DeviceGraph
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    rng = np.random.default_rng(9)
    off = np.arange(0, 6001, 30).astype(np.int64)
    g = DeviceGraph(0)
    for vmax in (300, 1_500_000_000, 300, 300, 70_000, 300):
        ids = (rng.integers(1, vmax + 1, off[-1]) * rng.choice([-1, 1], off[-1])).astype(np.int32)
        ids[:60] = np.tile(ids[:6], 10)
        g.build(ids, off, 5)
        assert O.diff_arrays(g.arrays(), c_oracle.COracleGraph(ids, off, 5).arrays()) == [], vmax
    g.close()


def test_gpu_k_sweep_on_resident_encoding():
    """EncodedReads keeps the CSR on the device; a k sweep over it equals building from the dict each time"""
    from amira_b200 import EncodedReads, GeneMerGraph, synth
    from tests.graph_snapshot import snapshot
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 800)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(synth.CONFIGS["c2"].vocab))
    enc = EncodedReads(reads)
    for k in (3, 5, 7):
        assert snapshot(GeneMerGraph(enc, k)) == snapshot(GeneMerGraph(reads, k))


def test_gpu_table_overflow_is_retried():
    """capacity hints far too small: the device reports the overflow and the build is redone larger"""
    from amira_b200 import synth
    from amira_b200.device_graph import DeviceGraph
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    ids, off = synth.generate(synth.CONFIGS["c3"], 0, 20000)
    ref = c_oracle.COracleGraph(ids, off, 3).arrays()
    g = DeviceGraph(0)
    for mask in (0, 3):                      # 16-byte bucketed tables, then the 32-byte ones
        g.debug_layout(mask)
        g.reserve(10, 10)
        g.build(ids, off, 3)
        assert O.diff_arrays(g.arrays(), ref) == [], mask
    g.close()


def test_gpu_random_small_inputs(dg):
    """hundreds of tiny random read sets over tiny vocabularies (tandem repeats, self edges, hairpins,
    palindromes, multi-edges, empty reads) -- the GPU build and both filters against the C oracle"""
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    from tests.test_random_small_cpu import random_reads
    n_pal = n_multi = 0
    for seed in range(300):
        rng = np.random.default_rng(1000 + seed)
        reads = random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        k = int(rng.integers(1, 6))
        vocab = O.build_vocabulary(reads)
        ids, off, _, _ = O.encode_reads(reads, vocab)
        try:
            ref = c_oracle.COracleGraph(ids, off, k)
        except AssertionError:
            n_pal += 1
            with pytest.raises(AssertionError):
                dg.build(ids, off, k)
            continue
        dg.build(ids, off, k)
        assert O.diff_arrays(dg.arrays(), ref.arrays()) == [], seed
        c = int(rng.integers(1, 5))
        try:
            ref.remove_low_coverage_components(c)
        except TypeError:
            n_multi += 1
            with pytest.raises(TypeError):
                dg.remove_low_coverage_components(c)
            continue
        dg.remove_low_coverage_components(c)
        assert O.diff_arrays(dg.arrays(), ref.arrays()) == [], seed
        a, b = int(rng.integers(1, 4)), int(rng.integers(1, 4))
        ref.filter_graph(a, b)
        dg.filter_graph(a, b)
        assert O.diff_arrays(dg.arrays(), ref.arrays()) == [], seed
    assert n_pal > 0 and n_multi >= 0


@pytest.mark.parametrize("out_of_place", [False, True])
@pytest.mark.parametrize("vmax", [40, 2_000_000, 2**31 - 2])
def test_gpu_segmented_sort_all_size_classes(dg, out_of_place, vmax):
    """the sort behind node -> reads / node -> edges: thread (<= 8), warp bitonic (<= 256), warp radix (<= 4096) and
    CTA radix (larger) segments, in place and out of place, with duplicates, against numpy"""
    rng = np.random.default_rng(11)
    sizes = np.concatenate([rng.integers(0, 10, 3000), rng.integers(0, 70, 2000), rng.integers(60, 520, 300),
                            [0, 1, 2, 8, 9, 31, 32, 33, 64, 65, 128, 129, 256, 257, 511, 512, 513, 1024, 1025, 4095, 4096,
                             4097, 5000, 16385, 40000, 70001], rng.integers(0, 10, 500)])
    rng.shuffle(sizes)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    data = rng.integers(0, vmax + 1, off[-1]).astype(np.uint32)
    small_range = rng.random(len(sizes)) < 0.3                      # many duplicates in some segments
    for s in np.flatnonzero(small_range):
        data[off[s]:off[s + 1]] %= 50
    got, dups, total = dg.debug_segsort(data, off, out_of_place=out_of_place, max_value=vmax + 1)
    want = data.copy()
    want_dups = np.zeros(len(sizes), np.uint32)
    for s in range(len(sizes)):
        seg = np.sort(data[off[s]:off[s + 1]])
        want[off[s]:off[s + 1]] = seg
        want_dups[s] = int(np.count_nonzero(seg[1:] == seg[:-1]))
    assert np.array_equal(got, want)
    assert np.array_equal(dups, want_dups) and total == int(want_dups.sum())


def heavy_node_reads():
    """20000 reads that all carry the core genes 1, 2, 3, 4 (every 7th twice, around gene 9) beside a random tail of
    genes 5..399 -> (ids, off)"""
    rng = np.random.default_rng(3)
    reads = []
    for i in range(20000):                                   # every read carries (1,2,3[,4]) -> nodes on 20000 reads
        tail = (rng.integers(5, 400, rng.integers(0, 6)) * rng.choice([-1, 1])).tolist()
        core = [1, 2, 3, 4]
        if i % 7 == 0:
            core = core + [9] + core                          # the same gene-mers twice on this read
        if i % 2:
            core = [-g for g in reversed(core)]
        reads.append(core + tail if i % 3 else tail + core)
    off = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.int64)
    ids = np.concatenate([np.asarray(r, np.int32) for r in reads])
    return ids, off


def test_gpu_repeated_genemers_and_heavy_nodes(dg):
    """a gene-mer twice on one read (duplicate incidences are removed, coverage counts both) and nodes that lie
    on more reads than a CTA sorts in shared memory"""
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    ids, off = heavy_node_reads()
    for k in (3, 5):
        ref = c_oracle.COracleGraph(ids, off, k)
        dg.build(ids, off, k)
        assert O.diff_arrays(dg.arrays(), ref.arrays()) == [], k
        ref.filter_graph(3, 2)
        dg.filter_graph(3, 2)
        assert O.diff_arrays(dg.arrays(), ref.arrays()) == [], k


def test_gpu_node_confined_to_a_narrow_read_range(dg):
    """the unit kernel cuts a long read list into equal-width READ ranges; a gene-mer that only occurs on a narrow
    range of reads overfills a few of them (beyond what the warp networks take) and goes through the any-size
    in-place sort.  Also a second heavy node spread over all reads beside it, and duplicates inside the range."""
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    rng = np.random.default_rng(11)
    R = 400_000
    body = rng.integers(10, 60000, (R, 3)).astype(np.int32) * rng.choice(np.array([-1, 1], np.int32), (R, 3))
    reads = [body[i].tolist() for i in range(R)]
    for i in range(3000):                      # (1,2,3) on reads 0..2999 only; twice on every 5th of them
        reads[i] = [1, 2, 3] + ([7, 1, 2, 3] if i % 5 == 0 else [])
    for i in range(0, R, 40):                  # (4,5,6) on every 40th read
        if i >= 3000:
            reads[i] = [4, 5, 6]
    off = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.int64)
    ids = np.concatenate([np.asarray(r, np.int32) for r in reads])
    ref = c_oracle.COracleGraph(ids, off, 3)
    dg.build(ids, off, 3)
    assert O.diff_arrays(dg.arrays(), ref.arrays()) == []


def test_gpu_key_width_boundary_values(dg):
    """ids at the edge of the remembered key width (|id| = 2^(b-1) - 2 fits, -(2^(b-1) - 1) and -2^(b-1) must not be
    packed with b bits): the handle first sees V = 14, then ids that only use the two values beyond"""
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    rng = np.random.default_rng(9)
    off = np.arange(0, 1201, 12).astype(np.int64)
    small = (rng.integers(1, 15, off[-1]) * rng.choice([-1, 1], off[-1])).astype(np.int32)
    for k in (3, 5):
        dg.build(small, off, k)
        assert O.diff_arrays(dg.arrays(), c_oracle.COracleGraph(small, off, k).arrays()) == []
        for vals in ([-15, -16, 2, 3], [-16, 16, 15, -15], [14, -14, 1], [-31, -32, 30, 2]):
            ids = rng.choice(np.asarray(vals, np.int32), off[-1]).astype(np.int32)
            ids[::12] = 1                                    # no palindromes at even k, some structure
            dg.build(ids, off, k)
            assert O.diff_arrays(dg.arrays(), c_oracle.COracleGraph(ids, off, k).arrays()) == [], (k, vals)


def test_gpu_repeated_resident_builds_replay_a_graph(dg):
    """the same device-resident CSR built again and again (the k sweep / rebuild loop): from the second repeat on the
    library replays a captured CUDA graph -- results must stay those of the oracle, also when k or the reads change
    in between and when a replayed build is followed by filters"""
    import torch
    from amira_b200 import synth
    from oracle import c_oracle
    from oracle import gmg_oracle as O
    ids, off = synth.generate(synth.CONFIGS["c2"], 0, 8000)
    ids2, off2 = synth.generate(synth.CONFIGS["c3"], 0, 6000)
    d = [torch.from_numpy(x).cuda() for x in (ids, off, ids2, off2)]
    torch.cuda.synchronize()
    ref = {3: c_oracle.COracleGraph(ids, off, 3).arrays(), 5: c_oracle.COracleGraph(ids, off, 5).arrays()}
    ref2 = c_oracle.COracleGraph(ids2, off2, 3)
    for k in (3, 3, 3, 3, 5, 5, 5, 3, 3, 3):
        dg.build(d[0], d[1], k, on_device=True, wait=False)
        assert O.diff_arrays(dg.arrays(), ref[k]) == [], k
    for rep in range(4):
        dg.build(d[2], d[3], 3, on_device=True, wait=False)
    assert O.diff_arrays(dg.arrays(), ref2.arrays()) == []
    ref2.remove_low_coverage_components(5)
    dg.remove_low_coverage_components(5)
    ref2.filter_graph(3, 1)
    dg.filter_graph(3, 1)
    assert O.diff_arrays(dg.arrays(), ref2.arrays()) == []
    for rep in range(3):                      # back-to-back replays without looking at the results in between
        dg.build(d[0], d[1], 3, on_device=True, wait=False)
    assert O.diff_arrays(dg.arrays(), ref[3]) == []
    # duplicate incidences: reading the results of each build removes them by swapping the read lists into the
    # second buffer pair, so a graph captured before that swap would write into the wrong buffers
    ids3, off3 = heavy_node_reads()
    d3 = [torch.from_numpy(x).cuda() for x in (ids3, off3)]
    torch.cuda.synchronize()
    ref3 = c_oracle.COracleGraph(ids3, off3, 3).arrays()
    for rep in range(5):
        dg.build(d3[0], d3[1], 3, on_device=True, wait=False)
        assert O.diff_arrays(dg.arrays(), ref3) == [], rep
