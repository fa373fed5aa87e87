"""Cleaning the reads of bubbles and tips until stable (GeneMerGraph.clean_until_stable) on fresh, unfiltered graphs:
C3 at k = 5 (500k reads, 10 % bad calls) and one bench shard of C5 (1.25M reads, k = 5), min_tip_length = 6, no gene
spared.  Per input, in one run:
  - the rounds until stable, each with its counts (bubbles, branches, branches replaced, tips, tips clipped, steps
    rewritten, steps clipped, reads changed, calls after) and the device time of its bubble policy
    (amira_gmg_bubble_policy, with the bubbles it computes), its tip policy (amira_gmg_tip_policy, with the tips), its
    pass (amira_gmg_clean_reads to device outputs, both passes) and the rebuild from the cleaned device CSR; every call
    ends in a device synchronise, so a host clock times it;
  - clean_until_stable() end to end on a fresh lazy graph (--reps times);
  - the same cleaning written with the existing methods (clip_compacted_tips, a rebuild, correct_compacted_bubbles, a
    rebuild, until neither changes a read), and whether it gives the same reads; it need not, as it clips and corrects
    on different graphs;
  - the device-to-host bytes and copies of one clean_until_stable() call, from a torch.profiler trace of a run of its
    own, against the same for the loop of existing methods; the final copy of the cleaned CSR is part of both, and
    its size, computed from the arrays, is given beside them.
Prints one JSON line per input, with the card's name and power limit (and writes them to --out if given).

    python scripts/clean_rounds_probe.py [--inputs c3,c5] [--reps 3] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.bubble_rounds_probe import d2h_traffic, synced  # noqa: E402
from scripts.unitigs_probe import INPUTS, gpu_name_and_power  # noqa: E402

MIN_TIP_LENGTH = 6


def composition(GeneMerGraph, g, k):
    """clip, rebuild, correct bubbles, rebuild, until a round changes no read -> (graph, reads, rounds)"""
    cur, e, n = g, None, 0
    for _ in range(30):
        n += 1
        e2 = cur.clip_compacted_tips(MIN_TIP_LENGTH)
        moved = bool(e2.tip_clipped.any())
        if moved:
            e, cur = e2, GeneMerGraph(e2, k)
        e2 = cur.correct_compacted_bubbles()
        if e2.branch_rewritten.any():
            e, cur, moved = e2, GeneMerGraph(e2, k), True
        if not moved:
            break
    return cur, e, n


def probe(name, reps, gpu):
    from amira_b200 import GeneMerGraph, encode, synth
    cfg_name, n_reads, k = INPUTS[name]
    cfg = synth.with_k(synth.CONFIGS[cfg_name], k)
    ids, off = synth.generate(cfg, 0, n_reads)
    reads = synth.to_read_dict(ids, off, synth.vocabulary_names(cfg.vocab))
    enc = encode.EncodedReads(reads)
    res = {"gpu": gpu, "input": "%s, %d reads, unfiltered" % (cfg.name, n_reads), "k": k, "calls": int(off[-1]),
           "min_tip_length": MIN_TIP_LENGTH}

    # the rounds, step by step on the handle
    g = GeneMerGraph(enc, k)
    h = g._require_device_state()
    h.sync()
    rounds, csr = [], None
    for r in range(30):
        n_rep, t_bub = synced(lambda: h.bubble_policy([]), h)
        n_clip, t_tip = synced(lambda: h.tip_policy(MIN_TIP_LENGTH, []), h)
        x, t_pass = synced(lambda: h.clean_reads(None, None, on_device=True), h)
        row = {"bubbles": h.bubble_counts()[0], "branches": len(x["branch_rewritten"]), "replaced": n_rep,
               "tips": len(x["tip_clipped"]), "tips_clipped": n_clip, "steps": int(x["branch_rewritten"].sum()),
               "steps_clipped": int(x["tip_clipped"].sum()), "reads": int(x["changed"].sum()), "calls": len(x["ids"]),
               "bubble_policy_s": t_bub, "tip_policy_s": t_tip, "pass_s": t_pass}
        if row["steps"] == 0 and row["steps_clipped"] == 0:
            rounds.append(row)
            break
        csr = x
        _, row["rebuild_s"] = synced(lambda: h.build(x["ids"], x["off"], k, on_device=True, n_calls=len(x["ids"])), h)
        rounds.append(row)
    res["rounds"] = rounds
    del g, csr

    t = []
    for _ in range(reps + 1):                                # the first call also reserves the buffers: not kept
        g = GeneMerGraph(enc, k)
        g._require_device_state().sync()
        t0 = time.perf_counter()
        graph, out = g.clean_until_stable(MIN_TIP_LENGTH)
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
    res["same_reads"] = bool(e is not None and e.reads == out.reads)
    res["reads_differing"] = 0 if e is None else sum(e.reads[r] != out.reads[r] for r in out.read_ids)
    del e

    g = GeneMerGraph(enc, k)
    g._require_device_state().sync()
    res["until_stable_d2h_bytes"], res["until_stable_d2h_copies"] = \
        d2h_traffic(lambda: g.clean_until_stable(MIN_TIP_LENGTH))
    g = GeneMerGraph(enc, k)
    g._require_device_state().sync()
    res["existing_methods_d2h_bytes"], res["existing_methods_d2h_copies"] = \
        d2h_traffic(lambda: composition(GeneMerGraph, g, k))
    # the size of the final CSR and its flags and counts, computed from the arrays (not measured): what one copy of
    # them to the host moves
    R, G = len(out.read_ids), len(out.ids)
    res["final_csr_bytes_computed"] = (8 * (R + 1) + 4 * G * (1 if out.pos_start is None else 3) + R
                                       + 4 * (len(out.branch_rewritten) + len(out.tip_clipped)))
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
