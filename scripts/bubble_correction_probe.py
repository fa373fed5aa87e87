"""Bubble read correction (amira_gmg_correct_bubble_reads, GeneMerGraph.correct_compacted_bubbles) on fresh,
unfiltered graphs: C3 at k = 5 (500k reads, 10 % bad calls) and one bench shard of C5 (1.25M reads, k = 5).  Per
input, in one run:
  - the device call on a fresh build with the popping policy's replace_with: its first call (the unitig ranking, the
    read paths and the bubbles included; sizes only), the same call again, and DeviceGraph.correct_bubble_reads() with
    the outputs on the device (both passes); every call synchronises, so a host clock times it;
  - correct_compacted_bubbles() end to end on a fresh lazy graph, and the rebuild from the corrected resident CSR;
  - the same correction on a graph marked host-edited (materialisation timed apart), and whether both agree;
  - the counts: bubbles, branches, reads and steps rewritten, and the bubbles left after one round of
    correct + rebuild.
Prints one JSON line per input, with the card's name and power limit (and writes them to --out if given).

    python scripts/bubble_correction_probe.py [--inputs c3,c5] [--reps 3] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.unitigs_probe import INPUTS, gpu_name_and_power  # noqa: E402


def timed(f):
    t0 = time.perf_counter()
    f()
    return time.perf_counter() - t0


def probe(name, reps, gpu):
    from amira_b200 import GeneMerGraph, _lib, encode, synth
    cfg_name, n_reads, k = INPUTS[name]
    cfg = synth.with_k(synth.CONFIGS[cfg_name], k)
    ids, off = synth.generate(cfg, 0, n_reads)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(cfg.vocab))
    enc = encode.EncodedReads(reads)
    res = {"gpu": gpu, "input": "%s, %d reads, unfiltered" % (cfg.name, n_reads), "k": k, "calls": int(off[-1])}

    g = GeneMerGraph(enc, k)
    h = g._require_device_state()
    bub, u = g.compacted_bubbles(), g.compacted_unitigs()
    rw = np.ascontiguousarray(g._bubble_winners(bub, u, np.zeros(len(u["node_unitig"]), bool)), np.int32)
    L = h._lib
    n = C.c_int64()

    def sizes():
        _lib.check(L.amira_gmg_correct_bubble_reads(h._h, rw.ctypes.data_as(C.c_void_p), C.byref(n), *[None] * 6, 0))

    t = {x: [] for x in ("first", "repeat", "fill_on_device")}
    for _ in range(reps + 1):                               # the first round also reserves the buffers: not kept
        h.build_resident(enc, k)                            # a new graph: nothing cached
        h.sync()
        t["first"].append(timed(sizes))
        t["repeat"].append(timed(sizes))
        t["fill_on_device"].append(timed(lambda: h.correct_bubble_reads(rw, on_device=True)))
    out = h.correct_bubble_reads(rw)
    res.update(bubbles=len(bub["source"]), branches=len(bub["branch_unitig"]), branches_replaced=int((rw >= 0).sum()),
               reads_rewritten=int(out["changed"].sum()), steps_rewritten=int(out["branch_rewritten"].sum()),
               calls_after=int(out["off"][-1]), **{"device_%s_s" % x: v[1:] for x, v in t.items()})
    del g

    lazy = GeneMerGraph(enc, k)
    lazy._require_device_state().sync()
    t0 = time.perf_counter()
    e = lazy.correct_compacted_bubbles()
    res["correct_lazy_s"] = time.perf_counter() - t0
    res["lazy_graph_stayed_lazy"] = bool(lazy.__dict__["_lazy"])
    t0 = time.perf_counter()
    rebuilt = GeneMerGraph(e, k)
    rebuilt._require_device_state().sync()
    res["rebuild_from_corrected_s"] = time.perf_counter() - t0
    res["bubbles_after_one_round"] = len(rebuilt.compacted_bubbles()["source"])
    del rebuilt

    host = GeneMerGraph(enc, k)
    res["host_materialise_s"] = timed(host._touch)
    t0 = time.perf_counter()
    e2 = host.correct_compacted_bubbles()
    res["correct_host_s"] = time.perf_counter() - t0
    res["same_result"] = bool(np.array_equal(e.ids, e2.ids) and np.array_equal(e.off, e2.off) and e.reads == e2.reads)
    del host, lazy
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--inputs", default="c3,c5")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    torch.cuda.init()
    gpu = gpu_name_and_power()
    lines = []
    for name in a.inputs.split(","):
        lines.append(json.dumps(probe(name, a.reps, gpu)))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
