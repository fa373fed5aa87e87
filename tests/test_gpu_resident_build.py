"""Builds from device CSRs whose offsets array has the address of an earlier one: the call count a build reuses from
the previous build belongs to that build's array only.  Through the public classes (two lazy graphs of equal read
count on the shared handle, a host build between them, the first one's reads freed before the second's are
uploaded) and through one device buffer refilled between builds, each graph checked against the C oracle's build."""
import gc

import numpy as np
import pytest

from oracle import c_oracle
from oracle import gmg_oracle as O

pytestmark = pytest.mark.gpu

K = 3


def inputs():
    """two read sets of 20 000 reads, the second with fewer calls"""
    from amira_b200 import synth
    a, b = synth.generate(synth.CONFIGS["c2"], 0, 20000), synth.generate(synth.CONFIGS["c3"], 0, 20000)
    assert len(a[1]) == len(b[1]) and b[1][-1] < a[1][-1]
    return a, b


def test_gpu_lazy_graphs_of_equal_read_count_on_the_shared_handle():
    import torch
    from amira_b200 import GeneMerGraph, encode, synth
    (ids_a, off_a), (ids_b, off_b) = inputs()
    names = lambda c: synth.vocabulary_names(synth.CONFIGS[c].vocab)
    a = encode.EncodedReads(synth.to_read_dict(ids_a, off_a, names("c2")))
    g = GeneMerGraph(a, K)
    assert g.get_total_number_of_nodes() > 0
    GeneMerGraph({"r": ["+a", "+b", "+c", "+d"]}, K)            # a build from host arrays on the same handle
    del g, a
    gc.collect()
    torch.cuda.synchronize()
    b = encode.EncodedReads(synth.to_read_dict(ids_b, off_b, names("c3")))
    gb = GeneMerGraph(b, K)
    want = c_oracle.COracleGraph(b.ids, b.off, K).arrays()
    assert O.diff_arrays(gb._require_device_state().arrays(), want) == []


def test_gpu_a_device_buffer_refilled_between_builds():
    """the same offsets and ids buffers, refilled with reads of fewer calls after a host build, then built again"""
    import torch
    from amira_b200.device_graph import DeviceGraph
    (ids_a, off_a), (ids_b, off_b) = inputs()
    d_ids = torch.empty(len(ids_a), dtype=torch.int32, device="cuda")
    d_off = torch.empty(len(off_a), dtype=torch.int64, device="cuda")

    def fill(ids, off):
        d_ids[:len(ids)].copy_(torch.from_numpy(ids))
        d_off.copy_(torch.from_numpy(off))
        torch.cuda.synchronize()

    want_a = c_oracle.COracleGraph(ids_a, off_a, K).arrays()
    want_b = c_oracle.COracleGraph(ids_b, off_b, K).arrays()
    dg = DeviceGraph(0)
    try:
        fill(ids_a, off_a)
        dg.build(d_ids, d_off, K, on_device=True)
        assert O.diff_arrays(dg.arrays(), want_a) == []
        dg.build(np.asarray([1, 2, 3, 4], np.int32), np.asarray([0, 4], np.int64), K)
        fill(ids_b, off_b)
        dg.build(d_ids, d_off, K, on_device=True)
        assert O.diff_arrays(dg.arrays(), want_b) == []
        dg.build(d_ids, d_off, K, on_device=True)              # the same array again: the count is reused
        assert O.diff_arrays(dg.arrays(), want_b) == []
    finally:
        dg.close()
