"""The reads grouped by their path through the generator's AMR genes (GeneMerGraph.gene_paths, amira_gmg_gene_paths) on
C3 at k = 5 (500k reads, 10 % bad calls) and one bench shard of C5 (1.25M reads, k = 5), on a fresh unfiltered graph
and after clean_until_stable(6).  Per input and graph, in one run:
  - counts: occurrences, complete occurrences, clusters, clusters with at least 5 members against the loci the
    generator inserted, and the partial occurrences assigned, ambiguous and unassigned;
  - the device time of a first call (its buffers already reserved by an earlier call on another graph) and of a cached
    call; each call ends in a device synchronise, so a host clock times it;
  - gene_paths() end to end on a lazy graph (from a fresh build of the same reads);
  - the numpy path on a host-edited graph of the first --host-reads reads.
Prints one JSON line per input, with the card's name and power limit (and writes them to --out if given).

    python scripts/gene_paths_probe.py [--inputs c3,c5] [--host-reads 20000] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.bubble_rounds_probe import synced  # noqa: E402
from scripts.unitigs_probe import INPUTS, gpu_name_and_power  # noqa: E402

MIN_TIP_LENGTH = 6


def counts(x, loci):
    partial = x["occ_flanks"] != 3
    members = np.diff(x["member_off"])
    return {"occurrences": len(x["occ_read"]), "complete": int((~partial).sum()), "clusters": len(x["n_complete"]),
            "clusters_5_members": int((members >= 5).sum()), "loci_inserted": loci,
            "partial_assigned": int((partial & (x["occ_cluster"] >= 0)).sum()),
            "partial_ambiguous": int((x["occ_cluster"] == -2).sum()),
            "partial_unassigned": int((x["occ_cluster"] == -1).sum())}


def timed(g, genes):
    """(first call, cached call) of gene_paths on the handle of lazy graph g, in seconds"""
    h = g._require_device_state()
    h.sync()
    ranks = sorted(set(g._gene_ranks(genes)))
    x, first = synced(lambda: h.gene_paths(ranks), h)
    _, cached = synced(lambda: h.gene_paths(ranks), h)
    return x, first, cached


def probe(name, host_reads, gpu):
    from amira_b200 import GeneMerGraph, encode, synth
    cfg_name, n_reads, k = INPUTS[name]
    cfg = synth.with_k(synth.CONFIGS[cfg_name], k)
    ids, off = synth.generate(cfg, 0, n_reads)
    names = synth.vocabulary_names(cfg.vocab)
    pool = synth._pool(cfg)
    genes = [names[r - 1] for r in pool.amr.tolist()]
    loci = int(pool.amr_loci.sum())
    enc = encode.EncodedReads(synth.to_read_dict(ids, off, names))
    res = {"gpu": gpu, "input": "%s, %d reads" % (cfg.name, n_reads), "k": k, "calls": int(off[-1]),
           "genes": len(genes), "min_tip_length": MIN_TIP_LENGTH}

    warm = GeneMerGraph(enc, k)                              # reserves the buffers: not timed
    warm.gene_paths(genes)
    del warm
    g = GeneMerGraph(enc, k)
    x, first, cached = timed(g, genes)
    res["fresh"] = {**counts(x, loci), "first_call_s": first, "cached_call_s": cached}
    g = GeneMerGraph(enc, k)
    g._require_device_state().sync()
    t0 = time.perf_counter()
    g.gene_paths(genes)
    res["fresh"]["end_to_end_lazy_s"] = time.perf_counter() - t0
    assert g.__dict__["_lazy"]
    del g

    clean, _ = GeneMerGraph(enc, k).clean_until_stable(MIN_TIP_LENGTH)
    x, first, cached = timed(clean, genes)
    res["cleaned"] = {**counts(x, loci), "first_call_s": first, "cached_call_s": cached}
    del clean

    sub = encode.EncodedReads(synth.to_read_dict(ids[:off[host_reads]], off[:host_reads + 1], names))
    hst = GeneMerGraph(sub, k)
    lazy_x = hst.gene_paths(genes)
    hst._touch()
    t0 = time.perf_counter()
    hx = hst.gene_paths(genes)
    res["host_path"] = {"reads": host_reads, "s": time.perf_counter() - t0,
                        "same_as_device": all(np.array_equal(hx[f], lazy_x[f]) for f in hx)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--inputs", default="c3,c5")
    ap.add_argument("--host-reads", type=int, default=20000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    torch.cuda.init()
    gpu = gpu_name_and_power()
    lines = []
    for name in a.inputs.split(","):
        lines.append(json.dumps(probe(name, a.host_reads, gpu)))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
