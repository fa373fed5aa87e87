"""Host-side mirror on a box without a GPU: the element classes, the encoder (through the C ABI's
host entry point), the library's exported symbols, and -- with the device replaced by a C-oracle
backed test double -- the materialisation of exported arrays into upstream-shaped objects."""
import ctypes
import os
import re

import numpy as np
import pytest

import amira_b200
from amira_b200 import _lib, construct_graph, encode
from amira_b200.construct_gene import Gene
from amira_b200.construct_gene_mer import GeneMer
from amira_b200.construct_read import Read
from tests.fake_device import OracleBackedDevice
from tests.graph_snapshot import check_small_cases, snapshot
from tests.helpers import ROOT, check_postbuild


@pytest.fixture()
def fake_device(monkeypatch):
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", OracleBackedDevice)


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "amira_gmg.h")).read()
    declared = set(re.findall(r"\b(amira_[a-z0-9_]+)\s*\(", hdr))
    declared.discard("amira_gmg")
    assert declared == set(_lib.EXPORTED)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert b"sm_100a" in lib.amira_version()


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(_lib.AmiraLibraryError, match="no CPU fallback"):
        amira_b200.DeviceGraph(0)
    with pytest.raises(_lib.AmiraLibraryError):
        amira_b200.GeneMerGraph({"r": ["+a", "+b", "+c"]}, 3)


def test_gene_parsing_contract():
    g = Gene("+gene 1")
    assert (g.get_name(), g.get_strand()) == ("gene_1", 1)
    assert Gene("-x").reverse_gene() == Gene("+x")
    assert Gene("-x").__hash__() == -Gene("+x").__hash__()
    for bad, msg in ((" ", "Gene information is missing"), ("x1", "Strand information missing for: x1"),
                     ("+", "Gene name information missing for: +")):
        with pytest.raises(AssertionError) as ei:
            Gene(bad)
        assert str(ei.value) == msg


def test_gene_mer_canonical_and_hash_symmetry():
    fwd = [Gene("+a"), Gene("-b"), Gene("+c")]
    rev = [Gene("-c"), Gene("+b"), Gene("-a")]
    a, b = GeneMer(fwd), GeneMer(rev)
    assert a == b and a.__hash__() == b.__hash__()
    assert a.get_geneMerDirection() == -b.get_geneMerDirection()
    assert a.get_canonical_geneMer() == b.get_canonical_geneMer()
    with pytest.raises(AssertionError, match="identical"):
        GeneMer([Gene("+a"), Gene("-a")])
    with pytest.raises(AssertionError, match="empty"):
        GeneMer([])


def test_read_window_counts():
    calls = ["+g%d" % i for i in range(6)]
    for k, n in ((1, 6), (2, 5), (3, 4), (6, 1), (7, 0)):
        gms, pos = Read("r", calls).get_geneMers(k)
        assert len(gms) == n and pos == [None] * n
    gms, pos = Read("r", calls, [(i * 10, i * 10 + 5) for i in range(6)]).get_geneMers(3)
    assert pos[0] == (0, 25) and pos[-1] == (30, 55)


def test_encoder_matches_rank_definition_and_errors():
    reads = {"r1": ["+b", "-a", "+c c"], "r2": [], "r3": ["-c_c"]}
    vocab = encode.Vocabulary(encode.collect_names(reads))
    assert vocab.names == sorted(["a", "b", "c_c"], key=lambda n: Gene("+" + n).__hash__())
    ids, off, ps, pe = encode.encode_reads(reads, vocab)
    rank = {n: i + 1 for i, n in enumerate(vocab.names)}
    assert ids.tolist() == [rank["b"], -rank["a"], rank["c_c"], -rank["c_c"]]
    assert off.tolist() == [0, 3, 3, 4] and ps is None
    for bad, msg in (("  ", "Gene information is missing"), ("a", "Strand information missing for: a"),
                     ("-", "Gene name information missing for: -")):
        with pytest.raises(AssertionError) as ei:
            encode.encode_reads({"r": ["+a", bad]}, vocab)
        assert str(ei.value).startswith(msg)
    ids, off, ps, pe = encode.encode_reads({"r": ["+a", "-b"]}, vocab, {"r": [[1, 5], [7, 9]]})
    assert ps.tolist() == [1, 7] and pe.tolist() == [5, 9]


def test_materialised_graph_matches_upstream_small_cases(fake_device, golden_small):
    check_small_cases(amira_b200.GeneMerGraph, golden_small, pytest)


def test_host_mutators_and_gml(fake_device, tmp_path):
    g = amira_b200.GeneMerGraph({"read1": ["+gene1", "-gene2", "+gene3", "-gene4"],
                                 "read2": ["+gene1", "-gene2", "+gene3", "-gene6"]}, 3)
    assert g.get_total_number_of_nodes() == 3 and g.get_total_number_of_edges() == 4
    first = next(g.all_nodes())
    assert g.get_degree(first) == 2 and len(g.get_all_neighbors(first)) == 2
    gml = g.generate_gml(str(tmp_path / "test_gml"), 3, 1, 1)
    assert gml[0] == "graph\t[" and gml[1] == "multigraph 1" and gml[-1] == "]"
    assert sum(e.startswith("\tnode") for e in gml) == 3 and sum(e.startswith("\tedge") for e in gml) == 4
    # single-object removal on the host, then the GPU filter must refuse the stale device copy
    g.remove_node(first)
    assert g.get_total_number_of_nodes() == 2 and g.get_total_number_of_edges() == 0
    assert g.get_readNodes()["read1"][0] is None and g.get_reads_to_correct() == {"read1", "read2"}
    with pytest.raises(RuntimeError, match="modified on the host"):
        g.filter_graph(2, 1)
    g.assign_component_ids()
    assert g.components() == [1, 2]


def test_second_graph_does_not_corrupt_first(fake_device):
    reads = {"r1": ["+a", "+b", "+c", "+d"], "r2": ["+a", "+b", "+c", "+e"], "r3": ["+a", "+b", "+c"]}
    g1 = amira_b200.GeneMerGraph(reads, 3)
    g2 = amira_b200.GeneMerGraph({"x": ["+p", "+q", "+r", "+s"]}, 3)
    g1.filter_graph(2, 1)          # handle is owned by g2 now: g1 transparently rebuilds its device copy
    assert g1.get_total_number_of_nodes() == 1
    assert g2.get_total_number_of_nodes() == 2
    g1.filter_graph(4, 1)
    assert g1.get_total_number_of_nodes() == 0 and g1.get_readNodes()["r3"] == [None]


def test_bind_upstream_runs_upstream_methods_on_our_build(fake_device, golden_small):
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip("upstream checkout not present (only in the build container)")
    cg = ref_harness.load()
    Bound = amira_b200.bind_upstream(cg)
    check_small_cases(Bound, golden_small, pytest)
    reads = {"r%d" % i: ["+a", "+b", "+c", "+d", "+e", "+f"] for i in range(3)}
    reads["q"] = ["-f", "-e", "-d", "-c", "-x"]
    ours, theirs = Bound(reads, 3), cg.GeneMerGraph(reads, 3)
    assert snapshot(ours) == snapshot(theirs)
    assert isinstance(next(ours.all_nodes()), cg.Node)
    # methods only upstream defines, running on the objects we materialised
    n0 = next(ours.all_nodes())
    t0 = next(theirs.all_nodes())
    assert ours.get_linear_path_for_node(n0) == theirs.get_linear_path_for_node(t0)
    assert ours.get_nodes_containing("c") == theirs.get_nodes_containing("c")
    ours.filter_graph(2, 1), theirs.filter_graph(2, 1)
    assert snapshot(ours) == snapshot(theirs)


def test_encoded_reads_reuse_and_binary_round_trip(fake_device, tmp_path, golden_small):
    """one parse of the gene-call strings serves every k; the binary form round-trips to the same graph"""
    from amira_b200 import EncodedReads
    case = next(c for c in golden_small if not c.get("raises") and len(c["reads"]) >= 2 and c["positions"])
    enc = EncodedReads(case["reads"], case["positions"])
    a = snapshot(amira_b200.GeneMerGraph(enc, case["k"]))
    assert a == snapshot(amira_b200.GeneMerGraph(case["reads"], case["k"], case["positions"])) == case["build"]
    enc.save(str(tmp_path / "calls.npz"))
    back = EncodedReads.load(str(tmp_path / "calls.npz"))
    assert back.reads == {r: [("+" if t[0] == "+" else "-") + t[1:].replace(" ", "_") for t in v]
                          for r, v in case["reads"].items()}
    assert snapshot(amira_b200.GeneMerGraph(back, case["k"]))["node_hashes"] == a["node_hashes"]
    for k in (1, 2, 3):                     # the sweep: same encoding, different gene-mer sizes
        try:
            g1, g2 = amira_b200.GeneMerGraph(enc, k), amira_b200.GeneMerGraph(case["reads"], k, case["positions"])
        except AssertionError:
            continue
        assert snapshot(g1) == snapshot(g2)


def test_bulk_keys_equal_hashlib_pickle():
    """csrc/host_keys.cpp restates pickle protocol 4 + SHA-256: every opcode width and sign case, all arities"""
    import hashlib
    import pickle
    import random
    lib = _lib.load()
    random.seed(7)
    vals = [0, 1, -1, 127, 128, 255, 256, -128, -129, -255, -256, 65535, 65536, 2**31 - 1, 2**31, -2**31, -2**31 - 1,
            2**32, -2**32, 2**63, -2**63, 2**255, -(2**255), 2**256 - 1, -(2**256 - 1), 2**247, -(2**247), 2**248 - 1, -(2**248)]
    vals += [random.getrandbits(random.choice([8, 16, 31, 32, 33, 64, 200, 255, 256])) * random.choice([1, -1]) for _ in range(500)]
    for arity in (0, 1, 2, 3, 4, 5, 15):
        tuples = [tuple(random.choice(vals) for _ in range(arity)) for _ in range(300)]
        mags = np.zeros((len(tuples), max(arity, 1), 32), np.uint8)
        neg = np.zeros((len(tuples), max(arity, 1)), np.int8)
        for i, t in enumerate(tuples):
            for j, v in enumerate(t):
                mags[i, j] = np.frombuffer(abs(v).to_bytes(32, "big"), np.uint8)
                neg[i, j] = v < 0
        out = np.zeros((len(tuples), 32), np.uint8)
        assert lib.amira_host_tuple_sha(mags.ctypes.data_as(ctypes.c_void_p), neg.ctypes.data_as(ctypes.c_void_p),
                                        len(tuples), arity, out.ctypes.data_as(ctypes.c_void_p)) == 0
        for i, t in enumerate(tuples):
            assert out[i].tobytes() == hashlib.sha256(pickle.dumps(t, protocol=4)).digest(), (arity, t)


def statistics_values(G=None):
    """-> label -> result of graph_utils.get_overall_mean_node_coverages / remove_junk_reads / get_valid_reads_only
    (the scans callers run right after a build) on a C3 sample; the coverages both from the exported incidence
    array and from the objects"""
    from amira_b200 import synth
    cfg = synth.CONFIGS["c3"]
    ids, off = synth.generate(cfg, 0, 400)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(cfg.vocab))
    positions = {r: [(10 * i, 10 * i + 9) for i in range(len(v))] for r, v in reads.items()}
    g = (G or amira_b200.GeneMerGraph)(reads, 3, positions)
    v = {"mean_node_coverages": amira_b200.get_overall_mean_node_coverages(g)}
    g._incidence_arrays = None
    v["mean_node_coverages_from_objects"] = amira_b200.get_overall_mean_node_coverages(g)
    g = amira_b200.GeneMerGraph(reads, 3, positions)
    g.filter_graph(3, 1)
    for rate in (0.8, 0.5, 0.99):
        v["junk_reads_%s" % rate] = g.remove_junk_reads(rate)
    v["valid_reads_only"] = g.get_valid_reads_only()
    v["filtered_mean_node_coverages"] = amira_b200.get_overall_mean_node_coverages(g)
    return v


def test_post_build_statistics_match_upstream(fake_device):
    """against the results of upstream's own implementations on upstream's own graph, stored as digests (see
    tests/test_postbuild.py); with the upstream package at hand, also through the class bound to it"""
    from oracle import ref_harness
    check_postbuild("statistics/c3_400", statistics_values())
    if ref_harness.available():
        check_postbuild("statistics/c3_400", statistics_values(amira_b200.bind_upstream(ref_harness.load())))


def test_encoded_reads_round_trip_and_incremental_update(tmp_path):
    reads = {"r1": ["+a", "-b", "+c", "+d"], "r2": ["-d", "+b"], "r3": [], "r4": ["+e", "+a", "-c"]}
    pos = {"r1": [[1, 2], [3, 4], [5, 6], [7, 8]], "r2": [], "r3": [], "r4": [[1, 9], [10, 19], [20, 29]]}
    enc = encode.EncodedReads(dict(reads), dict(pos))
    enc.save(str(tmp_path / "calls.npz"))
    back = encode.EncodedReads.load(str(tmp_path / "calls.npz"))
    assert back.reads == reads and back.ids.tolist() == enc.ids.tolist() and back.off.tolist() == enc.off.tolist()
    assert back.positions["r2"] == [] and back.positions["r1"] == [(1, 2), (3, 4), (5, 6), (7, 8)]
    # incremental re-encode: same arrays as a fresh encoding of the edited dict, known genes only -> spliced
    enc2 = encode.EncodedReads(dict(reads))
    upd = enc2.update({"r2": ["+a", "+a", "-e"], "r4": ["+b"]})
    fresh = encode.EncodedReads(dict(enc2.reads))
    assert upd.ids.tolist() == fresh.ids.tolist() and upd.off.tolist() == fresh.off.tolist()
    assert upd.vocab.names == fresh.vocab.names
    upd2 = upd.update({"r1": ["+zzz_new_gene", "-a"]})          # a new gene re-ranks the vocabulary
    fresh2 = encode.EncodedReads(dict(upd.reads))
    assert upd2.ids.tolist() == fresh2.ids.tolist() and upd2.vocab.names == fresh2.vocab.names
