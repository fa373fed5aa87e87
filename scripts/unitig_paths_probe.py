"""Unitig links and read paths (amira_gmg_unitig_links, amira_gmg_read_unitig_paths) on fresh, unfiltered graphs: C3 at
k = 5 (500k reads, 10 % bad calls) and one bench shard of C5 (1.25M reads, k = 5).  Per input, in one run:
  - each device call on a fresh build: its first call (the unitig ranking included, sizes only), the same call again
    (cached), the other call after it (the ranking cached), and DeviceGraph.unitig_links() / read_unitig_paths() on
    the cached results (both passes and the copies to the host); every call synchronises, so a host clock times it;
  - GeneMerGraph.compacted_links() and read_unitig_paths() end to end on a fresh lazy graph;
  - the host implementation on a graph marked host-edited (materialisation, index arrays from the objects and
    _readNodes, numpy), and whether it gives the same arrays;
  - windows against read steps, and edges against links.
Prints one JSON line per input, with the card's name and power limit (and writes them to --out if given).

    python scripts/unitig_paths_probe.py [--inputs c3,c5] [--reps 3] [--out FILE]"""
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
    n_links = C.c_int64()
    path_off = np.zeros(len(reads) + 1, np.int64)

    def links():
        _lib.check(L.amira_gmg_unitig_links(h._h, C.byref(n_links), *[None] * 6))

    def paths():
        _lib.check(L.amira_gmg_read_unitig_paths(h._h, path_off.ctypes.data_as(C.c_void_p), *[None] * 5))

    t = {x: [] for x in ("links_first", "links_cached", "paths_after_links", "paths_first", "paths_cached",
                         "links_after_paths", "links_export", "paths_export")}
    for _ in range(reps + 1):                               # the first round also reserves the buffers: not kept
        h.build_resident(enc, k)                            # a new graph: nothing cached
        h.sync()
        t["links_first"].append(timed(links))
        t["links_cached"].append(timed(links))
        t["paths_after_links"].append(timed(paths))
        h.build_resident(enc, k)
        h.sync()
        t["paths_first"].append(timed(paths))
        t["paths_cached"].append(timed(paths))
        t["links_after_paths"].append(timed(links))
        t["links_export"].append(timed(h.unitig_links))
        t["paths_export"].append(timed(h.read_unitig_paths))
    s = h.sizes()
    res.update(nodes=s["nodes"], edges=s["edges"], windows=s["windows"], short_reads=h.sizes_early()["short_reads"],
               links=int(n_links.value), steps=int(path_off[-1]),
               **{"device_%s_s" % x: v[1:] for x, v in t.items()})
    p = h.read_unitig_paths()
    res["longest_step"] = int(p["length"].max()) if len(p["length"]) else 0
    del g

    lazy = GeneMerGraph(enc, k)
    lazy._require_device_state().sync()
    t0 = time.perf_counter()
    got_l = lazy.compacted_links()
    res["compacted_links_lazy_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    got_p = lazy.read_unitig_paths()
    res["read_unitig_paths_lazy_s"] = time.perf_counter() - t0
    res["lazy_graph_stayed_lazy"] = bool(lazy.__dict__["_lazy"])
    del lazy

    host = GeneMerGraph(enc, k)
    res["host_materialise_s"] = timed(host._touch)
    t0 = time.perf_counter()
    want_l = host.compacted_links()
    res["host_compacted_links_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    want_p = host.read_unitig_paths()
    res["host_read_unitig_paths_s"] = time.perf_counter() - t0
    res["same_result"] = all(got.keys() == want.keys() and
                             all(np.array_equal(got[f], want[f]) and got[f].dtype == want[f].dtype for f in want)
                             for got, want in ((got_l, want_l), (got_p, want_p)))
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
