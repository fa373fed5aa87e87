"""Simple bubbles (amira_gmg_bubbles) and pop_compacted_bubbles on fresh, unfiltered graphs: C3 at k = 5 (500k reads,
10 % bad calls) and one bench shard of C5 (1.25M reads, k = 5).  Per input, in one run:
  - the device call on a fresh build: its first call (the unitig ranking and the read paths included, sizes only),
    the same call again (cached), and DeviceGraph.bubbles() on the cached result (both passes and the copies to the
    host); every call synchronises, so a host clock times it;
  - pop_compacted_bubbles() end to end on a fresh lazy graph, and whether the graph stays lazy;
  - the same on a graph marked host-edited (materialisation timed apart), and whether both remove the same hashes in
    the same order and leave the same unitigs;
  - the counts: bubbles, branches, nodes removed, reads marked for correction.
Prints one JSON line per input, with the card's name and power limit (and writes them to --out if given).

    python scripts/bubbles_probe.py [--inputs c3,c5] [--reps 3] [--out FILE]"""
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
    res = {"gpu": gpu, "input": "%s, %d reads, unfiltered" % (cfg.name, n_reads), "k": k}

    g = GeneMerGraph(enc, k)
    h = g._require_device_state()
    L = h._lib
    B, NB = C.c_int64(), C.c_int64()

    def sizes():
        _lib.check(L.amira_gmg_bubbles(h._h, C.byref(B), C.byref(NB), *[None] * 6))

    t = {x: [] for x in ("first", "cached", "export")}
    for _ in range(reps + 1):                               # the first round also reserves the buffers: not kept
        h.build_resident(enc, k)                            # a new graph: nothing cached
        h.sync()
        t["first"].append(timed(sizes))
        t["cached"].append(timed(sizes))
        t["export"].append(timed(h.bubbles))
    s = h.sizes()
    bub = h.bubbles()
    u = h.unitigs()
    ulen = np.diff(u["unitig_off"])[bub["branch_unitig"]]
    res.update(nodes=s["nodes"], edges=s["edges"], unitigs=len(u["circular"]), bubbles=int(B.value),
               branches=int(NB.value), branches_per_bubble_max=int(np.diff(bub["branch_off"]).max()) if B.value else 0,
               branch_nodes_mean=float(ulen.mean()) if len(ulen) else 0.0,
               **{"device_%s_s" % x: v[1:] for x, v in t.items()})
    del g

    lazy = GeneMerGraph(enc, k)
    lazy._require_device_state().sync()
    t0 = time.perf_counter()
    got = lazy.pop_compacted_bubbles()
    res["pop_lazy_s"] = time.perf_counter() - t0
    res["lazy_graph_stayed_lazy"] = bool(lazy.__dict__["_lazy"])
    res["nodes_removed"] = len(got)
    lazy_unitigs = lazy.compacted_unitigs()
    res["reads_marked_for_correction"] = len(lazy.get_reads_to_correct())   # materialises the lazy graph
    del lazy

    host = GeneMerGraph(enc, k)
    res["host_materialise_s"] = timed(host._touch)
    before = len(host.get_reads_to_correct())
    t0 = time.perf_counter()
    want = host.pop_compacted_bubbles()
    res["pop_host_s"] = time.perf_counter() - t0
    res["host_reads_marked_for_correction"] = len(host.get_reads_to_correct())
    res["reads_marked_before_pop"] = before
    res["same_result"] = got == want and all(np.array_equal(lazy_unitigs[f], v)
                                             for f, v in host.compacted_unitigs().items())
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
