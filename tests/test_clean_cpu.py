"""Cleaning the reads of bubbles and tips in one pass, and in rounds until stable, without a GPU: hand-made probes at
k = 3 and k = 1 (a middle substitution with a last-call error, clips at both ends with an edit, a spared gene, no bubble
and no tip, an empty read set); the rebuild from one pass against the graph of the intended reads; the product's host
implementation (GeneMerGraph._cleaned_reads_over through clean_compacted_reads) against clean_loop of
tests/clean_reference.py on lazy graphs through the test doubles and on host-edited graphs, after filters, trimming and
remove_node, with and without positions; clean_until_stable against clean_rounds_loop, its definition; the source
reads left untouched; save / load."""
import copy
import os

import numpy as np
import pytest

from amira_b200 import construct_graph, encode
from oracle import gmg_oracle as O
from tests.clean_reference import CleanDevice, clean_loop, clean_rounds_loop, graph_policies
from tests.fake_device import OracleBackedDevice
from tests.test_bubbles_cpu import error_reads
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES
from tests.tip_reference import TipPolicyDevice
from tests.unitig_path_reference import read_path_loop
from tests.unitig_reference import unitig_loop

FIELDS = ("ids", "off", "pos_start", "pos_end", "changed", "branch_rewritten", "tip_clipped")
LONG = ["+%s" % c for c in "abcdefghijkl"]


def rc(read):
    return [("-" if g[0] == "+" else "+") + g[1:] for g in read[::-1]]


@pytest.fixture
def fake_device(monkeypatch):
    """lazy graphs on the test double without the policies: served by the host implementation over its arrays"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", OracleBackedDevice)


@pytest.fixture
def policy_device(monkeypatch):
    """lazy graphs on the test double with both policies but no clean_reads: the host implementation cleans"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", TipPolicyDevice)


@pytest.fixture
def clean_device(monkeypatch):
    """lazy graphs on the test double with clean_reads, served by the loops"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", CleanDevice)


def same(x, y, fields=FIELDS, ctx=""):
    for f in fields:
        if x[f] is None or y[f] is None:
            assert x[f] is None and y[f] is None, (ctx, f)
            continue
        assert x[f].dtype == y[f].dtype, (ctx, f, x[f].dtype, y[f].dtype)
        assert np.array_equal(x[f], y[f]), (ctx, f, x[f], y[f])


def as_out(e):
    return {f: getattr(e, f) for f in FIELDS}


def expected(g, min_tip_length, genes={}):
    """clean_loop on graph g with the two policies of the loops"""
    src = g._source_encoded()
    if g._on_device():
        a = w = g._require_device_state().arrays()
    else:
        a, w = g._unitig_index_arrays(), g._read_index_arrays()
        rank = {n: i + 1 for i, n in enumerate(g._vocab.names)}
        w["node_key"] = np.asarray([[x.get_strand() * rank[x.get_name()] for x in n.get_canonical_geneMer()]
                                    for n in g._nodes.values()], np.int64).reshape(len(g._nodes), int(g._kmerSize))
    bub, rw, tips, clip = graph_policies(g, genes, min_tip_length)
    aw = {**a, **w}
    u = unitig_loop(a)
    p = read_path_loop(aw, u)
    return clean_loop(aw, u, bub, p, tips, src.ids, src.off, src.pos_start, src.pos_end, rw, clip)


def cleaned(reads, k, min_tip_length=None, genes={}, positions=None):
    """clean_compacted_reads on a lazy graph, checked against the loops"""
    g = construct_graph.GeneMerGraph(reads, k, positions)
    min_tip_length = k + 1 if min_tip_length is None else min_tip_length
    e = g.clean_compacted_reads(min_tip_length, genes)
    same(as_out(e), expected(g, min_tip_length, genes))
    assert g.__dict__["_lazy"]
    return e


def truth(n=5, read=LONG):
    return {"t%d" % i: read for i in range(n)}


def graph_summary(g):
    return ({h: n.get_node_coverage() for h, n in g.get_nodes().items()},
            {h: e.get_edge_coverage() for h, e in g.get_edges().items()})


ONE_PASS = [  # (error read, the read one pass makes of it, edits, clips)
    (LONG[:3] + ["+x"] + LONG[4:-1] + ["+y"], LONG[:-1], 1, 1),             # a middle substitution, a last-call error
    (["+y"] + LONG[1:5] + ["+x"] + LONG[6:-1] + ["+z"], LONG[1:-1], 1, 2),   # clips at both ends and an edit
]


@pytest.mark.parametrize("case", range(len(ONE_PASS)))
@pytest.mark.parametrize("backwards", [False, True])
def test_one_pass_edits_and_clips_a_read_and_the_rebuild_is_clean(fake_device, case, backwards):
    err, want, n_edit, n_clip = ONE_PASS[case]
    if backwards:
        err, want = rc(err), rc(want)
    reads = {**truth(), "e": err}
    e = cleaned(reads, 3)
    assert e.reads["e"] == want and e.changed.tolist() == [0] * 5 + [1]
    assert e.branch_rewritten.sum() == n_edit and e.tip_clipped.sum() == n_clip
    for r in truth():
        assert e.reads[r] is reads[r]
    g = construct_graph.GeneMerGraph(e, 3)
    ref = construct_graph.GeneMerGraph({**truth(), "e": want}, 3)
    assert graph_summary(g) == graph_summary(ref)
    assert len(g.compacted_tips()["tip_unitig"]) == 0 and len(g.compacted_bubbles()["source"]) == 0


def test_one_pass_at_k_1(fake_device):
    """a two-gene detour and a last-call error at k = 1: the detour is a two-node branch, the error a one-node tip"""
    err = LONG[:3] + ["+x", "+w"] + LONG[5:-1] + ["+y"]
    e = cleaned({**truth(), "e": err}, 1)
    assert e.reads["e"] == LONG[:-1] and e.branch_rewritten.sum() == 1 and e.tip_clipped.sum() == 1


def test_two_reads_one_edited_one_clipped(fake_device):
    e = cleaned({**truth(), "e1": LONG[:3] + ["+x"] + LONG[4:], "e2": rc(LONG[:-1] + ["+y"])}, 3)
    assert e.reads["e1"] == LONG and e.reads["e2"] == rc(LONG[:-1]) and e.changed.tolist() == [0] * 5 + [1, 1]


def test_a_spared_gene(fake_device):
    reads = {**truth(), "e": LONG[:3] + ["+x"] + LONG[4:-1] + ["+y"]}
    e = cleaned(reads, 3, genes={"y"})
    assert e.reads["e"] == LONG[:-1] + ["+y"] and e.tip_clipped.sum() == 0 and e.branch_rewritten.sum() == 1
    e = cleaned(reads, 3, genes={"x"})
    assert e.reads["e"] == LONG[:3] + ["+x"] + LONG[4:-1] and e.tip_clipped.sum() == 1 and e.branch_rewritten.sum() == 0


def test_no_bubble_and_no_tip(fake_device):
    reads = truth()
    for k in (1, 3):
        e = cleaned(reads, k)
        assert not e.changed.any() and e.reads == reads and len(e.branch_rewritten) == 0 and len(e.tip_clipped) == 0


def test_empty_read_set(fake_device):
    g = construct_graph.GeneMerGraph({}, 3)
    e = g.clean_compacted_reads(4)
    assert e.reads == {} and e.off.tolist() == [0] and len(e.ids) == 0
    assert len(e.branch_rewritten) == 0 and len(e.tip_clipped) == 0
    graph, reads = g.clean_until_stable(4)
    assert graph is g and reads.reads == {} and [r["steps"] for r in reads.rounds] == [0]


def test_positions_go_with_their_calls(fake_device):
    pos = lambda read: [(10 * i, 10 * i + 5) for i in range(len(read))]
    err = ["+y"] + LONG[1:5] + ["+x"] + LONG[6:-1] + ["+z"]
    reads = {**truth(), "e": err}
    positions = {r: pos(x) for r, x in reads.items()}
    e = cleaned(reads, 3, positions=positions)
    assert e.reads["e"] == LONG[1:-1] and e.positions["e"] == pos(err)[1:-1]
    assert e.positions["t0"] is positions["t0"]


def test_the_double_paths(policy_device, clean_device):
    """the lazy path through the handle's clean_reads (the loops) and through the policies with the host
    implementation"""
    reads = {**truth(), "e": LONG[:3] + ["+x"] + LONG[4:-1] + ["+y"], "f": rc(LONG[:-1] + ["+z"])}
    e = cleaned(reads, 3)
    assert e.reads["e"] == LONG[:-1] and e.reads["f"] == rc(LONG[:-1])


def test_clean_device_protocol(clean_device):
    reads = {**truth(), "e": LONG[:3] + ["+x"] + LONG[4:-1] + ["+y"]}
    g = construct_graph.GeneMerGraph(reads, 3)
    h = g._require_device_state()
    with pytest.raises(Exception):
        h.clean_reads(None, None)                            # no policy on these bubbles or tips
    h.bubble_policy()
    with pytest.raises(Exception):
        h.clean_reads(None, None)                            # no tip policy
    h.tip_policy(4)
    assert h.clean_reads(None, None)["changed"].tolist() == [0] * 5 + [1]
    NB, Q = h.bubble_counts()[1], h.tip_count()
    with pytest.raises(ValueError):
        h.clean_reads(np.zeros(NB, np.int64), None)          # a branch replaced by itself
    with pytest.raises(ValueError):
        h.clean_reads(None, np.full(Q, 2, np.uint8))
    x = h.clean_reads(np.full(NB, -1), np.zeros(Q, np.uint8))
    assert not x["changed"].any()
    with pytest.raises(Exception):
        h.clean_reads(None, None)                            # host arrays overwrote both held policies


def test_bad_policy_arrays_raise(fake_device):
    g = construct_graph.GeneMerGraph({**truth(), "e": LONG[:3] + ["+x"] + LONG[4:-1] + ["+y"]}, 3)
    a = g._require_device_state().arrays()
    u, src = g.compacted_unitigs(), g._source_encoded()
    bub, tips = g.compacted_bubbles(), g.compacted_tips()
    p = g._read_paths_over(a, a)
    NB, Q = len(bub["branch_unitig"]), len(tips["tip_unitig"])
    ok_rw, ok_clip = np.full(NB, -1), np.zeros(Q, np.uint8)
    for rw, clip in ((np.zeros(NB, np.int64), ok_clip), (ok_rw, np.full(Q, 2)), (ok_rw, np.zeros(Q + 1)),
                     (np.full(NB + 1, -1), ok_clip)):
        with pytest.raises(ValueError):
            construct_graph.GeneMerGraph._cleaned_reads_over(u, p, bub, tips, a, a["node_key"], rw, clip, src)


def edited_pair(seed, rng, reads, k, positions=None):
    """a lazy and a host-edited graph of the reads after the same filter or trim, the host one also after a
    remove_node for some seeds; None when the build or an edit refuses the input"""
    try:
        lazy = construct_graph.GeneMerGraph(reads, k, positions)
        hst = construct_graph.GeneMerGraph(reads, k, positions)
        ops = [[], [("filter_graph", (2, 1))], [("filter_graph", (1, 2))], [("remove_short_linear_paths", (3,))]][seed % 4]
        for g in (lazy, hst):
            for op, args in ops:
                getattr(g, op)(*args)
        hst._touch()
        if seed % 5 == 1 and len(hst.get_nodes()):
            objs = list(hst.get_nodes().values())
            hst.remove_node(objs[int(rng.integers(len(objs)))])
    except (AssertionError, TypeError):                        # palindromic window, a removal that meets a multi-edge
        return None
    return lazy, hst


def with_positions(reads, rng):
    return {r: [(int(s), int(s) + 7) for s in np.sort(rng.integers(0, 10 ** 6, len(x)))] for r, x in reads.items()}


@pytest.mark.parametrize("device", ["fake_device", "clean_device"])
def test_host_implementation_against_the_loop(request, device):
    """error reads and random reads, lazy (through the double) and host-edited, before and after filter_graph,
    remove_short_linear_paths and remove_node, with positions for some seeds, random min_tip_length and a gene"""
    request.getfixturevalue(device)
    n = n_both = n_edit = n_clip = 0
    for seed in range(240 if device == "fake_device" else 80):
        rng = np.random.default_rng(54000 + seed)
        reads = error_reads(rng, int(rng.integers(10, 40))) if seed % 3 else random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)),
                                                              int(rng.integers(1, 14)))
        k = int(rng.integers(1, 4))
        genes = {"x0"} if seed % 4 == 0 else {}
        min_tip_length = int(rng.integers(1, k + 3))
        pos = with_positions(reads, rng) if seed % 2 else None
        pair = edited_pair(seed, rng, reads, k, pos)
        if pair is None:
            continue
        for g in pair:
            x = g.clean_compacted_reads(min_tip_length, genes)
            same(as_out(x), expected(g, min_tip_length, genes), ctx=(seed, g._on_device()))
            if g is pair[0]:
                n_edit += int(x.branch_rewritten.any())
                n_clip += int(x.tip_clipped.any())
                n_both += int(x.branch_rewritten.any() and x.tip_clipped.any())
        n += 1
    assert n >= (160 if device == "fake_device" else 50) and n_edit >= 10 and n_clip >= 10 and n_both >= 5, \
        (n, n_edit, n_clip, n_both)


@pytest.mark.parametrize("name", FIXTURES)
def test_host_implementation_on_fixtures(fake_device, name):
    from tests.helpers import load_input, read_dict
    vocab, ids, off, ps, pe = load_input(name)
    reads, pos = read_dict(vocab, ids, off, ps, pe)
    for k in (1, 3, 5):
        try:
            g = construct_graph.GeneMerGraph(reads, k, pos)
        except AssertionError:
            continue
        same(as_out(g.clean_compacted_reads(k + 1)), expected(g, k + 1), ctx=(name, k))


def test_single_corrections_are_unchanged(fake_device):
    """correct_compacted_bubbles carries no tip_clipped and clip_compacted_tips no branch_rewritten, and each is the
    clean pass with the other policy switched off"""
    reads = {**truth(), "e": LONG[:3] + ["+x"] + LONG[4:-1] + ["+y"]}
    g = construct_graph.GeneMerGraph(reads, 3)
    b, t = g.correct_compacted_bubbles(), g.clip_compacted_tips(4)
    assert not hasattr(b, "tip_clipped") and not hasattr(t, "branch_rewritten")
    assert b.reads["e"] == LONG[:-1] + ["+y"] and t.reads["e"] == reads["e"][:-1]
    a = g._require_device_state().arrays()
    u, src = g.compacted_unitigs(), g._source_encoded()
    bub, rw, tips, clip = graph_policies(g, {}, 4)
    p = g._read_paths_over(a, a)
    none_rw, none_clip = np.full(len(rw), -1), np.zeros(len(clip), np.uint8)
    C = construct_graph.GeneMerGraph
    x = C._cleaned_reads_over(u, p, bub, tips, a, a["node_key"], rw, none_clip, src)
    y = C._corrected_reads_over(u, p, bub, a, a["node_key"], rw, src)
    same(x, y, ("ids", "off", "changed", "branch_rewritten"))
    x = C._cleaned_reads_over(u, p, bub, tips, a, a["node_key"], none_rw, clip, src)
    y = C._clipped_reads_over(u, p, tips, a, clip, src)
    same(x, y, ("ids", "off", "changed", "tip_clipped"))


# ---- rounds -----------------------------------------------------------------------------------------------------

def state(g):
    """what clean_until_stable must leave as it was"""
    arrays = g._require_device_state().arrays() if g._on_device() else \
        ({h: n.get_node_coverage() for h, n in g._nodes.items()}, {h: e.get_edge_coverage() for h, e in g._edges.items()})
    return g._device_ops, g._encoded, dict(g._reads), g._minNodeCoverage, g._minEdgeCoverage, arrays


def same_state(x, y):
    assert x[:5] == y[:5]
    if isinstance(x[5], dict):
        assert O.diff_arrays(x[5], y[5]) == []
    else:
        assert x[5] == y[5]


def until_stable(g, min_tip_length, max_rounds=30, genes={}, filt=None):
    """the product against clean_rounds_loop; returns (graph, reads)"""
    before = state(g)
    graph, reads = g.clean_until_stable(min_tip_length, max_rounds, genes, filt)
    assert graph is g or graph.__dict__["_lazy"]
    same_state(state(g), before)
    want_g, want_e, want_changed, want_rounds = clean_rounds_loop(g, min_tip_length, max_rounds, genes, filt)
    assert reads.rounds == want_rounds
    assert reads.reads == want_e.reads and reads.positions == want_e.positions
    for f in ("ids", "off", "pos_start", "pos_end"):
        x, y = getattr(reads, f), getattr(want_e, f)
        assert (x is None and y is None) or np.array_equal(x, y), f
    assert np.array_equal(reads.changed, want_changed)
    if want_g is g:
        assert graph is g
    else:
        assert graph is not g and graph._device_ops == want_g._device_ops
        assert O.diff_arrays(graph._arrays(), want_g._arrays()) == []
        assert np.array_equal(reads.branch_rewritten, want_e.branch_rewritten)
        assert np.array_equal(reads.tip_clipped, want_e.tip_clipped)
    return graph, reads


def test_rounds_on_probes(clean_device):
    # the start error of f makes the junction b c d, so e's substitution forms a simple bubble only once round 1 has
    # clipped it
    reads = {**truth(), "e": LONG[:3] + ["+x"] + LONG[4:-1] + ["+y"], "f": rc(["+z"] + LONG[1:])}
    graph, out = until_stable(construct_graph.GeneMerGraph(reads, 3), 4)
    assert out.reads["e"] == LONG[:-1] and out.reads["f"] == rc(LONG[1:])
    assert [(r["steps"], r["steps_clipped"]) for r in out.rounds] == [(0, 2), (1, 0), (0, 0)]
    assert out.rounds[-1]["steps"] == 0 and out.rounds[-1]["steps_clipped"] == 0
    assert len(graph.compacted_tips()["tip_unitig"]) == 0 and len(graph.compacted_bubbles()["source"]) == 0
    for max_rounds in (0, 1):
        graph, out = until_stable(construct_graph.GeneMerGraph(reads, 3), 4, max_rounds)
        assert len(out.rounds) == max_rounds
    graph, out = until_stable(construct_graph.GeneMerGraph(truth(), 3), 4)
    assert len(out.rounds) == 1 and not out.changed.any()


def test_rounds_sweep(clean_device):
    """error and random reads, lazy and host-edited, with a filter for some seeds, spared genes for others"""
    n = multi = 0
    for seed in range(60):
        rng = np.random.default_rng(55000 + seed)
        reads = error_reads(rng, int(rng.integers(10, 30))) if seed % 3 else \
            random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)), int(rng.integers(1, 14)))
        k = int(rng.integers(1, 4))
        filt = (1, 2) if seed % 4 == 1 else None
        genes = {"x0"} if seed % 5 == 2 else {}
        pos = with_positions(reads, rng) if seed % 2 else None
        pair = edited_pair(seed, rng, reads, k, pos)
        if pair is None:
            continue
        for g in pair:
            _, out = until_stable(g, k + 1, 30, genes, filt)
            multi += int(sum(r["steps"] + r["steps_clipped"] > 0 for r in out.rounds) >= 2)
        n += 1
    assert n >= 40 and multi >= 5, (n, multi)


def test_the_source_reads_are_left_untouched_and_save_load(clean_device, tmp_path):
    reads = {**truth(), "e": LONG[:3] + ["+x"] + LONG[4:-1] + ["+y"], "f": rc(["+z"] + LONG[1:])}
    src = encode.EncodedReads(reads)
    before = copy.deepcopy((src.reads, src.ids, src.off, src.read_ids, src.vocab.names))
    g = construct_graph.GeneMerGraph(src, 3)
    e = g.clean_compacted_reads(4)
    graph, r = g.clean_until_stable(4)
    after = (src.reads, src.ids, src.off, src.read_ids, src.vocab.names)
    assert all(np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y for x, y in zip(before, after))
    assert e.vocab is src.vocab and e.read_ids is src.read_ids and e.reads is not src.reads
    assert e.reads["e"] == LONG[:3] + ["+x"] + LONG[4:-1] and e.reads["f"] == rc(LONG[1:]) and e.reads["t0"] is reads["t0"]
    assert r.reads["e"] == LONG[:-1] and r.reads["f"] == rc(LONG[1:])
    for x in (e, r):
        x.save(str(tmp_path / "c.npz"))
        back = encode.EncodedReads.load(str(tmp_path / "c.npz"))
        assert back.reads == x.reads and np.array_equal(back.ids, x.ids) and np.array_equal(back.off, x.off)


UPSTREAM = os.environ.get("AMIRA_REFERENCE_ROOT", "/root/reference")


@pytest.mark.skipif(not os.path.isfile(os.path.join(UPSTREAM, "amira", "construct_graph.py")),
                    reason="upstream checkout not present")
def test_clean_methods_are_not_upstream_names():
    """bind_upstream overrides upstream's methods by name: the new methods must not replace one of upstream's"""
    import ast
    with open(os.path.join(UPSTREAM, "amira", "construct_graph.py")) as f:
        tree = ast.parse(f.read())
    cls = [c for c in tree.body if isinstance(c, ast.ClassDef) and c.name == "GeneMerGraph"]
    assert len(cls) == 1
    names = {f.name for f in cls[0].body if isinstance(f, (ast.FunctionDef, ast.AsyncFunctionDef))}
    assert names and not names & {"_unmarked", "_bubble_marks_over", "_fill_edits", "_tip_marks_over",
                                  "_cleaned_reads_over", "_rounds_until_stable", "clean_compacted_reads", "_clean",
                                  "_handle_clean", "clean_until_stable"}
