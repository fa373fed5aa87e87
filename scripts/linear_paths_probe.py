"""Linear walks and dead-end trimming on a fresh, unfiltered graph of noisy reads (C3 at k = 5 by default): the size
pass of amira_gmg_linear_walks over all 2N states, the walks from the tips, and remove_short_linear_paths(4) on the
host path (a graph marked host-edited: materialisation, _linear_steps, _walk) and on the device path, in one run.
Prints one JSON line (and writes it to --out if given).

    python scripts/linear_paths_probe.py [--reads 500000] [--k 5] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_name_and_power():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=500000)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from amira_b200 import GeneMerGraph, _lib, encode, synth
    from amira_b200.device_graph import _ptr

    torch.cuda.init()
    cfg = synth.with_k(synth.CONFIGS["c3"], a.k)
    ids, off = synth.generate(cfg, 0, a.reads)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(cfg.vocab))
    enc = encode.EncodedReads(reads)
    res = {"gpu": gpu_name_and_power(), "input": "%s, %d reads, unfiltered" % (cfg.name, a.reads), "k": a.k}

    # the primitive: size pass over all 2N states, walks from every tip (warm-up call first)
    g = GeneMerGraph(enc, a.k)
    h = g._require_device_state()
    n = h.sizes()["nodes"]
    deg = h.linear_steps()["degree"]
    tips = np.flatnonzero(deg == 1)
    res.update(nodes=int(n), tips=int(len(tips)))
    all_states = np.arange(2 * n, dtype=np.int32)
    tip_states = np.ascontiguousarray(np.stack([2 * tips, 2 * tips + 1], 1).ravel(), np.int32)
    woff = np.zeros(len(all_states) + 1, np.int64)
    L = h._lib
    for rep in range(3):                                    # the first call builds the jump table
        h.build_resident(enc, a.k)                          # a new graph: the table is computed again in every pass
        h.sync()
        t0 = time.perf_counter()
        _lib.check(L.amira_gmg_linear_walks(h._h, _ptr(all_states), len(all_states), 0, _ptr(woff), None))
        t_size = time.perf_counter() - t0
        t0 = time.perf_counter()
        toff, tnodes = h.linear_walks(tip_states)
        t_tips = time.perf_counter() - t0
    res.update(size_pass_all_states_s=t_size, all_states_output_nodes=int(woff[-1]), tip_walks_s=t_tips,
               tip_walk_nodes=int(len(tnodes)))
    del g

    # remove_short_linear_paths(4): host path, then device path, each on a fresh build of the same reads
    host = GeneMerGraph(enc, a.k)
    t0 = time.perf_counter()
    host._touch()
    want = host.remove_short_linear_paths(4)
    res["host_path_s"] = time.perf_counter() - t0
    del host
    dev = GeneMerGraph(enc, a.k)
    dev._require_device_state().sync()
    t0 = time.perf_counter()
    got = dev.remove_short_linear_paths(4)
    res["device_path_s"] = time.perf_counter() - t0
    res["removed"] = len(got)
    res["same_result"] = got == want
    res["device_graph_stayed_lazy"] = bool(dev.__dict__["_lazy"])
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
