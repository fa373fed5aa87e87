"""Unitigs (amira_gmg_unitigs) on fresh, unfiltered graphs: C3 at k = 5 (500k reads, 10 % bad calls) and one bench
shard of C5 (1.25M reads, k = 5).  Per input, in one run:
  - the device call on a fresh build: its first call (successors, ranking, numbering, sizes only), the same call again
    (cached), and DeviceGraph.unitigs() on the cached result (both calls and the copies to the host);
  - GeneMerGraph.compacted_unitigs() end to end on a fresh lazy graph;
  - the host implementation on a graph marked host-edited (materialisation, index arrays from the objects, numpy
    ranking), and whether it gives the same arrays.
Prints one JSON line per input, with the card's name and power limit (and writes them to --out if given).

    python scripts/unitigs_probe.py [--inputs c3,c5] [--reps 3] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

INPUTS = {"c3": ("c3", 500000, 5), "c5": ("c5", 1250000, 5)}


def gpu_name_and_power():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


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
    U = C.c_int64()
    first, cached, export = [], [], []
    for _ in range(reps):
        h.build_resident(enc, k)                            # a new graph: nothing cached
        h.sync()
        t0 = time.perf_counter()
        _lib.check(L.amira_gmg_unitigs(h._h, C.byref(U), *[None] * 10))
        first.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        _lib.check(L.amira_gmg_unitigs(h._h, C.byref(U), *[None] * 10))
        cached.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        dev = h.unitigs()
        export.append(time.perf_counter() - t0)
    s = h.sizes()
    lens = np.diff(dev["unitig_off"])
    res.update(nodes=s["nodes"], edges=s["edges"], unitigs=int(U.value), circular=int(dev["circular"].sum()),
               longest=int(lens.max()) if len(lens) else 0, internal_edges=int(dev["edge_internal"].sum()),
               device_first_call_s=first, device_cached_call_s=cached, device_unitigs_export_s=export)
    del g

    lazy = GeneMerGraph(enc, k)
    lazy._require_device_state().sync()
    t0 = time.perf_counter()
    got = lazy.compacted_unitigs()
    res["compacted_unitigs_lazy_s"] = time.perf_counter() - t0
    res["lazy_graph_stayed_lazy"] = bool(lazy.__dict__["_lazy"])
    del lazy

    host = GeneMerGraph(enc, k)
    t0 = time.perf_counter()
    host._touch()
    res["host_materialise_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    want = host.compacted_unitigs()
    res["host_compacted_unitigs_s"] = time.perf_counter() - t0
    res["same_result"] = all(np.array_equal(got[f], want[f]) and got[f].dtype == want[f].dtype for f in want) and \
        got.keys() == want.keys()
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
