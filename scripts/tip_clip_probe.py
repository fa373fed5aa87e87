"""Tip clipping (amira_gmg_tips, amira_gmg_tip_policy, amira_gmg_clip_tip_reads, GeneMerGraph.clip_compacted_tips) on
fresh, unfiltered graphs: C3 at k = 5 (500k reads, 10 % bad calls) and one bench shard of C5 (1.25M reads, k = 5), with
min_length = k + 1.  Per input, in one run:
  - each device call on a fresh build: its first call (the unitig ranking and the read paths included, for the tips;
    sizes only) and the same call again; the clip with the outputs on the device (both passes); every call
    synchronises, so a host clock times it;
  - the counts: tips, tips clipped, reads and steps clipped, and the tips left after one clip and a rebuild from the
    device CSR (given its call count);
  - clip_compacted_tips() end to end on a fresh lazy graph, and on a graph marked host-edited (materialisation timed
    apart), and whether both agree.
Prints one JSON line per input, with the card's name and power limit (and writes them to --out if given).

    python scripts/tip_clip_probe.py [--inputs c3,c5] [--reps 3] [--out FILE]"""
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
    from amira_b200.device_graph import DeviceGraph
    cfg_name, n_reads, k = INPUTS[name]
    cfg = synth.with_k(synth.CONFIGS[cfg_name], k)
    ids, off = synth.generate(cfg, 0, n_reads)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(cfg.vocab))
    enc = encode.EncodedReads(reads)
    res = {"gpu": gpu, "input": "%s, %d reads, unfiltered" % (cfg.name, n_reads), "k": k, "min_length": k + 1,
           "calls": int(off[-1])}

    h = DeviceGraph(0)
    L, n = h._lib, C.c_int64()
    calls = {"tips": lambda: _lib.check(L.amira_gmg_tips(h._h, C.byref(n), None, None, None, None)),
             "tip_policy": lambda: _lib.check(L.amira_gmg_tip_policy(h._h, k + 1, None, 0, C.byref(n), None)),
             "clip_tip_reads": lambda: _lib.check(L.amira_gmg_clip_tip_reads(h._h, None, C.byref(n), *[None] * 6, 0))}
    t = {"%s_%s" % (c, x): [] for c in calls for x in ("first", "repeat")}
    t["clip_fill_on_device"] = []
    for _ in range(reps + 1):                               # the first round also reserves the buffers: not kept
        for c, f in calls.items():
            h.build_resident(enc, k)                        # a new graph: nothing cached
            h.sync()
            if c == "clip_tip_reads":
                h.tip_policy(k + 1)                         # the policy (and with it the tips) is not timed here
            t[c + "_first"].append(timed(f))
            t[c + "_repeat"].append(timed(f))
        t["clip_fill_on_device"].append(timed(lambda: h.clip_tip_reads(None, on_device=True)))
    h.build_resident(enc, k)
    tips = h.tips()
    n_clipped = h.tip_policy(k + 1)
    out = h.clip_tip_reads(None, on_device=True)
    res.update(tips=len(tips["tip_unitig"]), tips_clipped=n_clipped, reads_clipped=int(out["changed"].sum()),
               steps_clipped=int(out["tip_clipped"].sum()), calls_after=len(out["ids"]),
               **{"device_%s_s" % x: v[1:] for x, v in t.items()})
    h2 = DeviceGraph(0)
    h2.build(out["ids"], out["off"], k, on_device=True, n_calls=len(out["ids"]))
    res["tips_after_one_clip"] = h2.tip_count()
    h2.close()
    h.close()
    del out

    lazy = GeneMerGraph(enc, k)
    lazy._require_device_state().sync()
    t0 = time.perf_counter()
    e = lazy.clip_compacted_tips(k + 1)
    res["clip_lazy_s"] = time.perf_counter() - t0
    res["lazy_graph_stayed_lazy"] = bool(lazy.__dict__["_lazy"])
    host = GeneMerGraph(enc, k)
    res["host_materialise_s"] = timed(host._touch)
    t0 = time.perf_counter()
    e2 = host.clip_compacted_tips(k + 1)
    res["clip_host_s"] = time.perf_counter() - t0
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
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
