"""The scans and edits Amira runs right after a build (SURVEY.md 8f): coverage statistics, junk / valid read
selection, gene look-ups, linear paths, dead-end removal, AMR-node pruning, GML.

The expected results are digests in tests/golden/postbuild.json (tests/record_postbuild.py writes them).  They were
recorded from the drop-in class of the commit at which these tests last compared it, live, with upstream's own
functions on upstream's own graph of the same reads; upstream's package is not part of this repository.  On CPU the
device is the oracle-backed test double (scans, paths, GML and the node removals); with `-m gpu` everything runs on
the real device."""
import os

import pytest

import amira_b200
from amira_b200 import construct_graph, graph_utils
from tests.fake_device import OracleBackedDevice
from tests.graph_snapshot import snapshot
from tests.helpers import check_postbuild, load_input, read_dict

CASES = [("fixture_eight", 3), ("fixture_seven", 3), ("fixture_four", 5), ("synth_c2_2000", 3)]


def genes_of_interest(vocab):
    names = [n for n in vocab]
    return [names[i] for i in range(0, len(names), max(1, len(names) // 7))][:6] + ["not_a_gene_in_this_sample"]


def readonly_values(name, k, tmp):
    """-> (graph, vocabulary, label -> result of every read-only scan)"""
    vocab, ids, off, ps, pe = load_input(name)
    reads, pos = read_dict(vocab, ids, off, ps, pe)
    ours = amira_b200.GeneMerGraph({r: list(v) for r, v in reads.items()}, k, pos)
    v = {}
    # statistics straight from the device arrays (nothing materialised yet)
    assert ours.__dict__["_lazy"]
    v["overall_mean_node_coverages"] = graph_utils.get_overall_mean_node_coverages(ours)
    v["mean_node_coverage"] = ours.get_mean_node_coverage()
    v["all_node_coverages"] = ours.get_all_node_coverages()
    v["total_number_of_nodes"] = ours.get_total_number_of_nodes()
    v["components"] = ours.components()
    assert ours.__dict__["_lazy"], "the statistics must not need the host objects"
    # GML from the arrays
    out = os.path.join(str(tmp), "gml_%s_%d" % (name, k))
    v["gml_1_1"] = ours.generate_gml(out, k, 1, 1)
    assert ours.__dict__["_lazy"]
    # filters on the device, then the read selections (still no host objects)
    ours.filter_graph(3, 1)
    for er in (0.0, 0.2, 0.5, 0.93):
        v["junk_reads_%s" % er] = ours.remove_junk_reads(er)
    v["valid_reads_only"] = ours.get_valid_reads_only()
    v["gml_3_1"] = ours.generate_gml(out, k, 3, 1)
    assert ours.__dict__["_lazy"]
    v["snapshot_filtered"] = snapshot(ours)            # materialises from the filtered device graph
    # gene look-ups and linear paths
    for g in genes_of_interest(vocab):
        v["nodes_containing_" + g] = [n.__hash__() for n in ours.get_nodes_containing(g)]
    v["AMR_nodes"] = list(ours.get_AMR_nodes(genes_of_interest(vocab)))
    for want in (False, True):
        v["linear_paths_%s" % want] = [ours.get_linear_path_for_node(n, want) for n in ours.all_nodes()]
    return ours, vocab, v


def edit_values(ours, vocab):
    """dead ends: remove_short_linear_paths (construct_graph.py:679-720) with and without genes of interest, then
    pruning to the reads of the genes of interest"""
    v = {}
    v["short_paths_4"] = sorted(ours.remove_short_linear_paths(4, genes_of_interest(vocab)[:2]))
    v["snapshot_short_paths_4"] = snapshot(ours)
    v["short_paths_6"] = sorted(ours.remove_short_linear_paths(6))
    v["snapshot_short_paths_6"] = snapshot(ours)
    ours.remove_non_AMR_associated_nodes(genes_of_interest(vocab))
    v["snapshot_non_AMR_removed"] = snapshot(ours)
    return v


def k_sweep_values():
    """choose_kmer_size's sweep (graph_utils.py:258-296): one encoding, resident CSR, one build per k"""
    vocab, ids, off, ps, pe = load_input("fixture_four")
    reads, pos = read_dict(vocab, ids, off, ps, pe)
    v = {}
    for k, g in graph_utils.build_k_sweep(reads, range(3, 10, 2), pos).items():
        assert g.__dict__["_lazy"]
        v["k%d_mean_node_coverage" % k] = g.get_mean_node_coverage()
        v["k%d_snapshot" % k] = snapshot(g)
    return v


def lazy_rebuild_values():
    """a graph whose device copy was overwritten by a later build (one handle per device) rebuilds and replays its
    device operations before answering"""
    vocab, ids, off, ps, pe = load_input("fixture_eight")
    reads, pos = read_dict(vocab, ids, off, ps, pe)
    g1 = amira_b200.GeneMerGraph(reads, 3)
    g1.remove_low_coverage_components(5)
    g1.filter_graph(3, 1)
    g2 = amira_b200.GeneMerGraph(reads, 5)
    return {"g1_mean_node_coverage": g1.get_mean_node_coverage(), "g1_snapshot": snapshot(g1),
            "g2_total_number_of_nodes": g2.get_total_number_of_nodes()}


@pytest.fixture()
def fake_device(monkeypatch):
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", OracleBackedDevice)


@pytest.mark.parametrize("name,k", CASES[:2])
def test_postbuild_scans_cpu_double(fake_device, tmp_path, name, k):
    check_postbuild("scans/%s_k%d" % (name, k), readonly_values(name, k, tmp_path)[2])


@pytest.mark.parametrize("name,k", CASES[:2])
def test_postbuild_edits_cpu_double(fake_device, tmp_path, name, k):
    """the node removals (linear-path pruning, AMR pruning) through the test double's remove_nodes /
    remove_nodes_without_reads_of, against the digests the device recorded"""
    ours, vocab, v = readonly_values(name, k, tmp_path)
    check_postbuild("scans/%s_k%d" % (name, k), v)
    check_postbuild("edits/%s_k%d" % (name, k), edit_values(ours, vocab))


@pytest.mark.gpu
@pytest.mark.parametrize("name,k", CASES)
def test_postbuild_scans_gpu(tmp_path, name, k):
    ours, vocab, v = readonly_values(name, k, tmp_path)
    check_postbuild("scans/%s_k%d" % (name, k), v)
    check_postbuild("edits/%s_k%d" % (name, k), edit_values(ours, vocab))


@pytest.mark.gpu
def test_k_sweep_on_resident_reads_gpu():
    check_postbuild("k_sweep/fixture_four", k_sweep_values())


@pytest.mark.gpu
def test_lazy_graph_survives_another_build_gpu():
    check_postbuild("lazy_rebuild/fixture_eight", lazy_rebuild_values())
