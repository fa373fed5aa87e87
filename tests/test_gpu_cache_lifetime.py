"""How long the post-build caches and the held policies live: until the next build, filter or node removal on their
handle, and no shorter.  A build on another handle, a policy call with many gene ranks, or a walk query larger than
any before it leaves the cached tables and the held policies of a handle in place; a filter or a removal of no node
ends them."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K = 5


@pytest.fixture(scope="module")
def c3():
    from amira_b200 import synth
    return synth.generate(synth.CONFIGS["c3"], 0, 20000)


@pytest.fixture
def new_graph():
    from amira_b200.device_graph import DeviceGraph
    made = []

    def make(ids, off):
        g = DeviceGraph(0)
        made.append(g)
        return g.build(ids, off, K)

    yield make
    for g in made:
        g.close()


def exports(g):
    return {"unitigs": g.unitigs(), "links": g.unitig_links(), "paths": g.read_unitig_paths(), "bubbles": g.bubbles(),
            "tips": g.tips()}


def same(x, y, ctx):
    assert x.keys() == y.keys(), ctx
    for f in x:
        if x[f] is None or y[f] is None:
            assert x[f] is None and y[f] is None, (ctx, f)
        elif isinstance(x[f], dict):
            same(x[f], y[f], (ctx, f))
        else:
            assert np.array_equal(x[f], y[f]), (ctx, f)


def held_status(g):
    """the status of correct_bubble_reads and clip_tip_reads with the held policies (size passes)"""
    L, n = g._lib, C.c_int64()
    return (L.amira_gmg_correct_bubble_reads(g._h, None, C.byref(n), *[None] * 6, 0),
            L.amira_gmg_clip_tip_reads(g._h, None, C.byref(n), *[None] * 6, 0))


def test_gpu_caches_and_policies_survive_a_build_on_another_handle(c3, new_graph):
    from amira_b200 import synth
    a = new_graph(*c3)
    want = exports(a)
    a.bubble_policy((5,))
    a.tip_policy(K + 1)
    corrected, clipped = a.correct_bubble_reads(None), a.clip_tip_reads(None)
    assert corrected["changed"].any() and clipped["changed"].any()
    n = a.kernel_launches()
    b = new_graph(*synth.generate(synth.CONFIGS["c3"], 1, 60000))   # a larger graph: every buffer of b grows
    b.tips()
    same(exports(a), want, "exports after the build on another handle")
    assert a.kernel_launches() == n                                   # nothing recomputed
    same(a.correct_bubble_reads(None), corrected, "held replace_with")
    same(a.clip_tip_reads(None), clipped, "held clip flags")


@pytest.mark.parametrize("tips_first", [True, False])
def test_gpu_a_held_policy_survives_the_other_policy_with_many_gene_ranks(c3, new_graph, tips_first):
    """the other family's policy call grows the room for gene ranks: 100 000 ranks, all but one absent from the
    vocabulary"""
    g = new_graph(*c3)
    many = np.concatenate([[5], np.arange(10**6, 10**6 + 99999)]).astype(np.int32)
    if tips_first:
        g.tip_policy(K + 1)
        want = g.clip_tip_reads(None)
        g.bubble_policy(many)
        same(g.clip_tip_reads(None), want, "clip flags held across bubble_policy")
    else:
        g.bubble_policy((5,))
        want = g.correct_bubble_reads(None)
        g.tip_policy(K + 1, many)
        same(g.correct_bubble_reads(None), want, "replace_with held across tip_policy")
    assert want["changed"].any()


def test_gpu_the_walk_table_survives_a_larger_query(c3, new_graph):
    g = new_graph(*c3)
    deg = g.linear_steps()["degree"]
    ends = np.flatnonzero(deg == 1)[:32]
    small = np.stack([2 * ends, 2 * ends + 1], 1).ravel()
    deltas, want = [], None
    for _ in range(3):
        n = g.kernel_launches()
        want = g.linear_walks(small)
        deltas.append(g.kernel_launches() - n)
    # the first query builds the table, and the ones after it, its output included, keep it
    assert len(want[1]) > 0 and deltas[0] > deltas[1] == deltas[2], deltas
    big = g.linear_walks(np.tile(small, 4000))                        # more states and more output than before
    assert len(big[1]) == 4000 * len(want[1])
    n = g.kernel_launches()
    got = g.linear_walks(small)
    assert g.kernel_launches() - n == deltas[1]
    assert all(np.array_equal(x, y) for x, y in zip(got, want))


@pytest.mark.parametrize("change", ["filter_graph", "remove_nodes"])
def test_gpu_a_filter_or_removal_ends_the_caches_and_policies(c3, new_graph, change):
    from amira_b200 import _lib
    g = new_graph(*c3)
    g.bubble_policy((5,))
    g.tip_policy(K + 1)
    exports(g)
    assert held_status(g) == (_lib.OK, _lib.OK)
    if change == "filter_graph":
        g.filter_graph(1, 1)                                          # keeps every node, and is a new graph all the same
    else:
        g.remove_nodes(np.zeros(g.sizes()["nodes"], np.uint8))
    for name, f in (("unitigs", g.unitigs), ("links", g.unitig_links), ("paths", g.read_unitig_paths),
                    ("bubbles", g.bubbles), ("tips", g.tips)):
        n = g.kernel_launches()
        f()
        assert g.kernel_launches() > n, name                          # recomputed
    assert g.bubble_counts()[1] > 0 and g.tip_count() > 0
    assert held_status(g) == (_lib.E_STATE, _lib.E_STATE)
