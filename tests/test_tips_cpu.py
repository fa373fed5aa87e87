"""Tip clipping without a GPU: hand-made probes with known answers at k = 3 and k = 1 (a substitution at the last, the
second-last and the first call in both read orientations, a deletion and a strand flip at a read end, one-node tips of
both orientations, two tips on one junction, a tip whose mean equals its sibling's, a tip of min_length nodes, a spared
gene, a read lying wholly on a tip, a read clipped at both ends, a tip step followed by None windows after a filter, a
self edge next to a dead end, a tip off a circle); the rebuild from the clipped reads against the build of the
truncated reads; the product's host implementation (GeneMerGraph._tips_over, _tip_clip_flags, _clipped_reads_over)
against the loops of tests/tip_reference.py on lazy graphs through the test doubles and on host-edited graphs, after
filters, trimming and remove_node; positions; the source reads left untouched; save / load."""
import copy
import os

import numpy as np
import pytest

from amira_b200 import construct_graph, encode
from oracle import gmg_oracle as O
from tests.bubble_rounds_reference import spared_nodes
from tests.fake_device import OracleBackedDevice
from tests.test_bubbles_cpu import TRUE, error_reads
from tests.test_random_small_cpu import random_reads
from tests.test_unitigs_cpu import FIXTURES
from tests.tip_reference import TipDevice, TipPolicyDevice, clip_loop, reference_tips, tip_loop, tip_policy_loop
from tests.unitig_path_reference import read_path_loop
from tests.unitig_reference import unitig_loop

FIELDS = ("ids", "off", "pos_start", "pos_end", "changed", "tip_clipped")
TIP_FIELDS = ("tip_unitig", "tip_orient", "tip_attach", "tip_reads")


def rc(read):
    return [("-" if g[0] == "+" else "+") + g[1:] for g in read[::-1]]


@pytest.fixture
def fake_device(monkeypatch):
    """lazy graphs on the test double without the tip calls: served by the host implementation over its arrays"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", OracleBackedDevice)


@pytest.fixture
def tip_device(monkeypatch):
    """lazy graphs on the test double with tips() only: the policy and the clip by the host implementation"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", TipDevice)


@pytest.fixture
def loop_device(monkeypatch):
    """lazy graphs on the test double with every tip call, served by the loops"""
    monkeypatch.setattr(construct_graph, "_HANDLES", {})
    monkeypatch.setattr(construct_graph, "DeviceGraph", TipPolicyDevice)


def same(x, y, fields=FIELDS, ctx=""):
    for f in fields:
        if x[f] is None or y[f] is None:
            assert x[f] is None and y[f] is None, (ctx, f)
            continue
        assert x[f].dtype == y[f].dtype, (ctx, f, x[f].dtype, y[f].dtype)
        assert np.array_equal(x[f], y[f]), (ctx, f, x[f], y[f])


def as_out(e):
    return {f: getattr(e, f) for f in FIELDS}


def graph_arrays(g):
    """the arrays the loops read for graph g: a lazy graph's device arrays, or a host-edited graph's objects"""
    if g._on_device():
        a = g._require_device_state().arrays()
        return a, a
    return g._unitig_index_arrays(), g._read_index_arrays()


def expected(g, min_length, genes={}):
    """(tips, clip flags, clipped reads) of graph g by the loops"""
    src = g._source_encoded()
    a, w = graph_arrays(g)
    if g._on_device():
        amr = spared_nodes(a, g._gene_ranks(list(genes)))
    else:
        amr_nodes = g.get_AMR_nodes(genes)
        amr = np.asarray([nh in amr_nodes for nh in g._nodes], bool)
    aw = {**a, **w}
    u = unitig_loop(a)
    p = read_path_loop(aw, u)
    tips = tip_loop(a, u, p)
    clip = tip_policy_loop(a, u, tips, amr, min_length)
    return tips, clip, clip_loop(aw, u, p, tips, src.ids, src.off, src.pos_start, src.pos_end, clip)


def clipped(reads, k, min_length=None, genes={}, positions=None):
    """clip_compacted_tips on a lazy graph, checked against the loops"""
    g = construct_graph.GeneMerGraph(reads, k, positions)
    min_length = k + 1 if min_length is None else min_length
    tips, _, want = expected(g, min_length, genes)
    same(g.compacted_tips(), tips, TIP_FIELDS)
    e = g.clip_compacted_tips(min_length, genes)
    same(as_out(e), want)
    assert g.__dict__["_lazy"]
    return e


def graph_summary(g):
    return ({h: n.get_node_coverage() for h, n in g.get_nodes().items()},
            {h: e.get_edge_coverage() for h, e in g.get_edges().items()})


def truth(n=5):
    return {"t%d" % i: TRUE for i in range(n)}


SINGLE = [  # (error read, the read it is clipped to)
    (TRUE[:-1] + ["+x"], TRUE[:-1]),                         # the last call
    (TRUE[:-2] + ["+x", "+g"], TRUE[:-2]),                   # the second-last call
    (["+x"] + TRUE[1:], TRUE[1:]),                           # the first call
    (TRUE[:-2] + ["+g"], TRUE[:-2]),                         # a deletion at the read end
    (TRUE[:-1] + ["-g"], TRUE[:-1]),                         # a strand flip at the read end
]


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("case", range(len(SINGLE)))
@pytest.mark.parametrize("backwards", [False, True])
def test_one_end_error_is_clipped_and_the_rebuild_has_no_tip(fake_device, k, case, backwards):
    err, want = SINGLE[case]
    if k == 1 and case in (1, 3, 4):                         # at k = 1 these make a bubble, an edge or the same node
        pytest.skip("no tip at k = 1")
    if backwards:
        err, want = rc(err), rc(want)
    reads = {**truth(), "e": err}
    e = clipped(reads, k)
    assert e.reads["e"] == want and e.changed.tolist() == [0] * 5 + [1], (e.reads["e"], want)
    assert e.tip_clipped.sum() == 1 and not hasattr(e, "branch_rewritten")
    for r in truth():
        assert e.reads[r] is reads[r]
    g = construct_graph.GeneMerGraph(e, k)
    ref = construct_graph.GeneMerGraph({**truth(), "e": want}, k)
    assert graph_summary(g) == graph_summary(ref)
    assert len(g.compacted_tips()["tip_unitig"]) == 0


def test_the_true_end_is_a_tip_kept_by_its_coverage(fake_device):
    g = construct_graph.GeneMerGraph({**truth(), "e": TRUE[:-1] + ["+x"]}, 3)
    tips = g.compacted_tips()
    assert len(tips["tip_unitig"]) == 2 and sorted(tips["tip_reads"].tolist()) == [1, 5]
    assert len(set(tips["tip_attach"].tolist())) == 1
    tips, clip, _ = expected(g, 4)
    assert sorted(zip(tips["tip_reads"].tolist(), clip.tolist())) == [(1, 1), (5, 0)]


def test_one_node_tips_of_both_orientations(fake_device):
    """one-node tips entered from either side of their node: the orientation follows which state is dead"""
    seen = set()
    for err in (TRUE[:-1] + ["+x"], TRUE[:-1] + ["-x"], ["+x"] + TRUE[1:], ["-x"] + TRUE[1:]):
        for read in (err, rc(err)):
            reads = {**truth(), "e": read}
            e = clipped(reads, 3)
            assert len(e.reads["e"]) == 6 and e.changed.tolist() == [0] * 5 + [1]
            g = construct_graph.GeneMerGraph(reads, 3)
            tips, clip, _ = expected(g, 4)
            seen |= set(tips["tip_orient"][clip == 1].tolist())
    assert seen == {1, -1}


def test_two_tips_on_one_junction(fake_device):
    e = clipped({**truth(), "e1": TRUE[:-1] + ["+x"], "e2": TRUE[:-1] + ["+y"]}, 3)
    assert e.reads["e1"] == TRUE[:-1] and e.reads["e2"] == TRUE[:-1] and e.tip_clipped.tolist().count(1) == 2


def test_a_tip_whose_mean_equals_its_siblings_is_kept(fake_device):
    e = clipped({"t": TRUE, "e": TRUE[:-1] + ["+x"]}, 3)
    assert not e.changed.any() and e.tip_clipped.tolist() == [0, 0]


def test_a_tip_of_min_length_nodes_is_kept(fake_device):
    reads = {**truth(), "e": TRUE[:-2] + ["+x", "+g"]}              # a tip of two nodes
    assert not clipped(reads, 3, min_length=2).changed.any()
    assert clipped(reads, 3, min_length=3).reads["e"] == TRUE[:-2]


def test_a_tip_with_a_gene_of_interest_is_spared(fake_device):
    reads = {**truth(), "e": TRUE[:-1] + ["+x"]}
    e = clipped(reads, 3, genes={"x"})
    assert not e.changed.any() and e.reads == reads
    assert clipped(reads, 3, genes={"q"}).reads["e"] == TRUE[:-1]


def test_a_read_wholly_on_a_tip_is_left_alone(fake_device):
    reads = {**truth(), "e": TRUE[:-1] + ["+x"], "w": ["+e", "+f", "+x"]}
    e = clipped(reads, 3)
    assert e.reads["e"] == TRUE[:-1] and e.reads["w"] is reads["w"] and e.changed.tolist() == [0] * 5 + [1, 0]


def test_a_read_clipped_at_both_ends(fake_device):
    for read in (["+y"] + TRUE[1:-1] + ["+x"], rc(["+y"] + TRUE[1:-1] + ["+x"])):
        e = clipped({**truth(), "e": read}, 3)
        assert e.reads["e"] == read[1:-1] and e.tip_clipped.sum() == 2


def test_a_tip_step_followed_by_none_windows(fake_device):
    """filter_graph(2, 2) removes x y z (one read): the step of e2 on the tip no longer reaches its read's end"""
    reads = {**truth(), "e1a": TRUE[:-1] + ["+x", "+y"], "e1b": TRUE[:-1] + ["+x", "+y"],
             "e2": TRUE[:-1] + ["+x", "+y", "+z"]}
    g = construct_graph.GeneMerGraph(reads, 3)
    g.filter_graph(2, 2)
    tips, clip, want = expected(g, 4)
    assert clip.sum() == 1
    e = g.clip_compacted_tips(4)
    same(as_out(e), want)
    assert e.changed.tolist() == [0] * 5 + [1, 1, 0] and e.reads["e1a"] == TRUE[:-1] and e.reads["e2"] is reads["e2"]


def test_a_self_edge_next_to_a_dead_end(fake_device):
    reads = {**truth(), "e": TRUE + ["+x", "+x"]}
    g = construct_graph.GeneMerGraph(reads, 1)
    tips = g.compacted_tips()
    u = g.compacted_unitigs()
    (key,) = g._arrays("node_key")
    xs = set(u["node_unitig"][np.flatnonzero(np.abs(key[:, 0]) == g._gene_ranks(["x"])[0])].tolist())
    assert not xs & set(tips["tip_unitig"].tolist())
    clipped(reads, 1)


def test_a_tip_off_a_circle(fake_device):
    loop = ["+a", "+b", "+c", "+d", "+e", "+f", "+g", "+a", "+b", "+c"]
    e = clipped({**{"t%d" % i: loop for i in range(4)}, "e": loop[:8] + ["+x"]}, 3)
    assert e.reads["e"] == loop[:8] and e.changed.tolist() == [0] * 4 + [1]


def test_positions_go_with_their_calls(fake_device):
    pos = lambda read: [(10 * i, 10 * i + 5) for i in range(len(read))]
    reads = {**truth(), "e": ["+y"] + TRUE[1:-2] + ["+x", "+g"]}
    positions = {r: pos(x) for r, x in reads.items()}
    e = clipped(reads, 3, positions=positions)
    assert e.reads["e"] == TRUE[1:-2] and e.positions["e"] == pos(reads["e"])[1:-2]
    assert e.positions["t0"] is positions["t0"]


def test_the_source_reads_are_left_untouched_and_save_load(fake_device, tmp_path):
    reads = {**truth(), "e": TRUE[:-1] + ["+x"], "f": rc(["+x"] + TRUE[1:])}
    src = encode.EncodedReads(reads)
    before = copy.deepcopy((src.reads, src.ids, src.off, src.read_ids, src.vocab.names))
    g = construct_graph.GeneMerGraph(src, 3)
    e = g.clip_compacted_tips(4)
    after = (src.reads, src.ids, src.off, src.read_ids, src.vocab.names)
    assert all(np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y for x, y in zip(before, after))
    assert g._encoded is src and e.vocab is src.vocab and e.read_ids is src.read_ids and e.reads is not src.reads
    assert e.reads["e"] == TRUE[:-1] and e.reads["f"] == rc(TRUE[1:]) and e.reads["t0"] is reads["t0"]
    e.save(str(tmp_path / "c.npz"))
    back = encode.EncodedReads.load(str(tmp_path / "c.npz"))
    assert back.reads == e.reads and np.array_equal(back.ids, e.ids) and np.array_equal(back.off, e.off)


def test_device_double_paths(tip_device):
    """tips() from the double, the policy and the clip by the host implementation"""
    e = clipped({**truth(), "e": TRUE[:-1] + ["+x"], "f": rc(["+x"] + TRUE[1:])}, 3)
    assert e.reads["e"] == TRUE[:-1] and e.reads["f"] == rc(TRUE[1:])


def test_loop_device_path(loop_device):
    """the lazy path through the double's tip_policy / clip_tip_reads gives the same as the host implementation"""
    e = clipped({**truth(), "e": TRUE[:-1] + ["+x"], "f": rc(TRUE[:-2] + ["+x", "+g"])}, 3)
    assert e.reads["e"] == TRUE[:-1] and e.reads["f"] == rc(TRUE[:-2])
    g = construct_graph.GeneMerGraph({**truth(), "e": TRUE[:-1] + ["+x"]}, 3)
    h = g._require_device_state()
    with pytest.raises(Exception):
        h.clip_tip_reads(None)                               # no policy on these tips
    assert h.tip_policy(4) == 1
    assert h.clip_tip_reads(None)["changed"].tolist() == [0] * 5 + [1]


def edited_pair(seed, rng, reads, k):
    """a lazy and a host-edited graph of the reads, after the same filter or trim, the host one also after a
    remove_node for some seeds; None when the build or an edit refuses the input"""
    try:
        lazy = construct_graph.GeneMerGraph(reads, k)
        hst = construct_graph.GeneMerGraph(reads, k)
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


def test_host_implementation_against_the_loops(fake_device):
    """error reads and random reads, lazy and host-edited, before and after filter_graph, remove_short_linear_paths
    and remove_node; random min_length and a gene of interest"""
    n = n_changed = n_tips = 0
    for seed in range(300):
        rng = np.random.default_rng(51000 + seed)
        reads = error_reads(rng) if seed % 3 else random_reads(rng, int(rng.integers(1, 25)), int(rng.integers(2, 9)),
                                                              int(rng.integers(1, 14)))
        k = int(rng.integers(1, 4))
        genes = {"x0"} if seed % 4 == 0 else {}
        min_length = int(rng.integers(1, k + 3))
        pair = edited_pair(seed, rng, reads, k)
        if pair is None:
            continue
        for g in pair:
            tips, _, want = expected(g, min_length, genes)
            same(g.compacted_tips(), tips, TIP_FIELDS, (seed, g._on_device()))
            x = g.clip_compacted_tips(min_length, genes)
            same(as_out(x), want, ctx=(seed, g._on_device()))
            if g is pair[0]:
                n_changed += int(x.changed.any())
                n_tips += len(tips["tip_unitig"])
        n += 1
    assert n >= 200 and n_changed >= 30 and n_tips >= 250, (n, n_changed, n_tips)


def test_min_length_k_plus_one_on_error_reads(fake_device):
    """min_length = k + 1 on error reads at k = 1 and 3: every clipped read keeps k calls or more (clip_loop asserts
    it), and the counts are those the loops give"""
    tips = clipped_tips = changed = 0
    for seed in range(150):
        for k in (1, 3):
            rng = np.random.default_rng(52000 + seed)
            reads = error_reads(rng)
            try:
                g = construct_graph.GeneMerGraph(reads, k)
            except AssertionError:
                continue
            t, clip, want = expected(g, k + 1)
            e = g.clip_compacted_tips(k + 1)
            same(as_out(e), want, ctx=(seed, k))
            tips += len(t["tip_unitig"])
            clipped_tips += int(clip.sum())
            changed += int(e.changed.sum())
    assert tips >= 200 and clipped_tips >= 100 and changed >= 100, (tips, clipped_tips, changed)


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
        tips, _, want = expected(g, k + 1)
        same(g.compacted_tips(), tips, TIP_FIELDS, (name, k))
        same(as_out(g.clip_compacted_tips(k + 1)), want, ctx=(name, k))


def test_empty_graph(fake_device):
    g = construct_graph.GeneMerGraph({}, 3)
    assert len(g.compacted_tips()["tip_unitig"]) == 0
    e = g.clip_compacted_tips(4)
    assert e.reads == {} and e.off.tolist() == [0] and len(e.ids) == 0 and len(e.tip_clipped) == 0


def test_bad_clip_flags_raise():
    reads = {**truth(), "e": TRUE[:-1] + ["+x"]}
    vocab = O.build_vocabulary(reads)
    ids, off, _, _ = O.encode_reads(reads, vocab)
    dev = TipPolicyDevice().build(ids, off, 3)
    a = dev.arrays()
    u, p, tips = reference_tips(a)
    src = encode.EncodedReads(reads)
    for clip in ([0, 2], [1], [0, 0, 0], [-1, 0]):
        with pytest.raises(ValueError):
            dev.clip_tip_reads(np.asarray(clip))
        with pytest.raises(ValueError):
            construct_graph.GeneMerGraph._clipped_reads_over(u, p, tips, a, np.asarray(clip), src)


def test_bubble_results_are_unchanged_by_the_shared_tail(fake_device):
    """correct_compacted_bubbles still carries branch_rewritten and no tip_clipped"""
    e = construct_graph.GeneMerGraph({**truth(), "e": ["+a", "+b", "+c", "+x", "+e", "+f", "+g"]}, 3) \
        .correct_compacted_bubbles()
    assert e.reads["e"] == TRUE and e.branch_rewritten.tolist() == [0, 1] and not hasattr(e, "tip_clipped")


UPSTREAM = os.environ.get("AMIRA_REFERENCE_ROOT", "/root/reference")


@pytest.mark.skipif(not os.path.isfile(os.path.join(UPSTREAM, "amira", "construct_graph.py")),
                    reason="upstream checkout not present")
def test_tip_methods_are_not_upstream_names():
    """bind_upstream overrides upstream's methods by name: the new methods must not replace one of upstream's"""
    import ast
    with open(os.path.join(UPSTREAM, "amira", "construct_graph.py")) as f:
        tree = ast.parse(f.read())
    cls = [c for c in tree.body if isinstance(c, ast.ClassDef) and c.name == "GeneMerGraph"]
    assert len(cls) == 1
    names = {f.name for f in cls[0].body if isinstance(f, (ast.FunctionDef, ast.AsyncFunctionDef))}
    assert names and not names & {"compacted_tips", "_tips_over", "_tip_clip_flags", "_clipped_reads_over",
                                  "clip_compacted_tips", "_tip_clip", "_untouched_calls_over"}
