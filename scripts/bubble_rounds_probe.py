"""Correcting the reads through the simple bubbles until none is left (GeneMerGraph.correct_bubbles_until_stable) on
fresh, unfiltered graphs: C3 at k = 5 (500k reads, 10 % bad calls) and one bench shard of C5 (1.25M reads, k = 5).
Per input, in one run:
  - the rounds until stable, each with its counts (bubbles left, branches, branches replaced, steps and reads
    rewritten, calls after) and the device time of its policy (amira_gmg_bubble_policy, with the bubbles it computes),
    its correction (amira_gmg_correct_bubble_reads to device outputs, both passes) and the rebuild from the corrected
    device CSR; every call ends in a device synchronise, so a host clock times it;
  - correct_bubbles_until_stable() end to end on a fresh lazy graph (--reps times);
  - the same loop written with the existing methods (correct_compacted_bubbles, then GeneMerGraph(reads, k)), and
    whether both give the same reads;
  - the device-to-host bytes and copies of one whole call, from a torch.profiler trace of a run of its own, against
    the same for the loop of existing methods; the final copy of the corrected CSR is part of both.
Prints one JSON line per input, with the card's name and power limit (and writes them to --out if given).

    python scripts/bubble_rounds_probe.py [--inputs c3,c5] [--reps 3] [--out FILE]"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.unitigs_probe import INPUTS, gpu_name_and_power  # noqa: E402


def synced(f, h):
    t0 = time.perf_counter()
    x = f()
    h.sync()
    return x, time.perf_counter() - t0


def composition(GeneMerGraph, g, k):
    cur, e, n = g, None, 0
    for _ in range(30):
        e2 = cur.correct_compacted_bubbles()
        n += 1
        if not e2.branch_rewritten.any():
            break
        e, cur = e2, GeneMerGraph(e2, k)
    return cur, e, n


def d2h_traffic(f):
    """(bytes, copies) device to host during f(), from a CUDA-activity trace"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    copies = [e for e in events if e.get("cat") == "gpu_memcpy" and "DtoH" in e.get("name", "")]
    return int(sum(e.get("args", {}).get("bytes", 0) for e in copies)), len(copies)


def probe(name, reps, gpu):
    from amira_b200 import GeneMerGraph, encode, synth
    cfg_name, n_reads, k = INPUTS[name]
    cfg = synth.with_k(synth.CONFIGS[cfg_name], k)
    ids, off = synth.generate(cfg, 0, n_reads)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(cfg.vocab))
    enc = encode.EncodedReads(reads)
    res = {"gpu": gpu, "input": "%s, %d reads, unfiltered" % (cfg.name, n_reads), "k": k, "calls": int(off[-1])}

    # the rounds, step by step on the handle
    g = GeneMerGraph(enc, k)
    h = g._require_device_state()
    h.sync()
    rounds, csr = [], None
    for r in range(30):
        n_rep, t_pol = synced(lambda: h.bubble_policy([]), h)
        x, t_cor = synced(lambda: h.correct_bubble_reads(None, on_device=True), h)
        B, NB = h.bubble_counts()
        row = {"bubbles": B, "branches": NB, "replaced": n_rep, "steps": int(x["branch_rewritten"].sum()),
               "reads": int(x["changed"].sum()), "calls": len(x["ids"]), "policy_s": t_pol, "correct_s": t_cor}
        if row["steps"] == 0:
            rounds.append(row)
            break
        csr = x
        _, row["rebuild_s"] = synced(lambda: h.build(x["ids"], x["off"], k, on_device=True), h)
        rounds.append(row)
    res["rounds"] = rounds
    del g, csr

    t = []
    for _ in range(reps + 1):                                # the first call also reserves the buffers: not kept
        g = GeneMerGraph(enc, k)
        g._require_device_state().sync()
        t0 = time.perf_counter()
        graph, out = g.correct_bubbles_until_stable()
        graph._require_device_state().sync()
        t.append(time.perf_counter() - t0)
        del g, graph
    res["until_stable_s"] = t[1:]
    res["until_stable_rounds"] = out.rounds
    res["changed_reads"] = int(out.changed.sum())

    t = []
    for _ in range(reps):
        g = GeneMerGraph(enc, k)
        g._require_device_state().sync()
        t0 = time.perf_counter()
        cur, e, n = composition(GeneMerGraph, g, k)
        cur._require_device_state().sync()
        t.append(time.perf_counter() - t0)
        del g, cur
    res["existing_methods_s"] = t
    res["existing_methods_rounds"] = n
    res["same_result"] = bool(e is not None and np.array_equal(e.ids, out.ids) and np.array_equal(e.off, out.off)
                              and e.reads == out.reads)
    del e

    g = GeneMerGraph(enc, k)
    g._require_device_state().sync()
    res["until_stable_d2h_bytes"], res["until_stable_d2h_copies"] = d2h_traffic(lambda: g.correct_bubbles_until_stable())
    g = GeneMerGraph(enc, k)
    g._require_device_state().sync()
    res["existing_methods_d2h_bytes"], res["existing_methods_d2h_copies"] = \
        d2h_traffic(lambda: composition(GeneMerGraph, g, k))
    R, G = len(out.read_ids), len(out.ids)
    res["final_csr_d2h_bytes"] = 8 * (R + 1) + 4 * G + R + 4 * len(out.branch_rewritten)
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
