#!/usr/bin/env python
"""bench.py -- gene-mers/s of the GeneMerGraph build on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # upstream's own Python path on the host CPU

Workload (config.workload): the C5 metagenome-scale synthetic gene-call set of BASELINE.json
(configs[4]: 10M reads x 30 gene calls, 60k-gene vocabulary, 50 genomes, 1% bad calls, k=5), weak-scaled:
every GPU builds over its contiguous shard of 1.25M reads, so N=8 is the full 10M-read set and N=1 is
one shard (37.4M gene calls, 32.4M gene-mers; 150 MB of gene ids, larger than the 126 MB L2).

A step = one complete build of the graph of the resident reads: window enumeration,
canonicalisation, node/edge hash tables, first-seen ordering, per-read node lists, node->read
incidence, adjacency, connected components -- everything GeneMerGraph.__init__ computes
(upstream amira/construct_graph.py:31-102).

  value    gene-mers/s with the CSR input already resident in HBM (CUDA events on the handle's stream; builds are
           enqueued back to back, the library does not synchronise with the host during a build)
  e2e      the same through the C ABI with HOST buffers: pinned host CSR -> amira_gmg_build (H2D inside)
           -> every graph array exported back to pinned host memory (D2H inside)
  parity   the graph of the timed workload, digested field by field and compared with the C oracle's digests of the
           same input (tests/golden/bench_digests.json; live oracle run for non-default sizes); FAIL -> exit code 3
  roofline / cpu_baseline / clocks: see DESIGN.md "Measurement"
  extras   the other BASELINE.json configs on one GPU (C2 with CUDA-graph replay, C3 k=3/5/7 through the filters,
           C4), each with its own parity check

One JSON line on stdout (rank 0).  Everything else goes to stderr.

--dump-outputs DIR writes the graph arrays of the last timed build (rank 0's, as a caller of DeviceGraph.arrays()
receives them) to DIR/<name>.npy; the workload is seeded, so two builds of the project can be compared array by array.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from dataclasses import replace

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

READS_PER_GPU = 1_250_000
METRIC = "gene-mers/sec GeneMerGraph build"
UNIT = "gene-mers/s"
BYTES_PER_GENE_MER = 13          # SURVEY.md 8(d): 4 id in + 4 node idx + 1 direction + 4 node->read incidence out
ATOMICS_PER_GENE_MER = 3         # SURVEY.md 8(d): 1 node update + 2 directed-edge updates
DIGESTS = os.path.join(ROOT, "tests", "golden", "bench_digests.json")

_REAL_STDOUT = None


def emit(obj):
    """the one JSON line, on the process's original stdout"""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def workload(n_gpus: int, rank: int, reads_per_gpu: int):
    from amira_b200 import synth
    cfg = replace(synth.CONFIGS["c5"], n_reads=reads_per_gpu * n_gpus)
    ids, off = synth.generate(cfg, rank * reads_per_gpu, reads_per_gpu)
    return cfg, ids, off


def config_dict(cfg, n_gpus, reads_per_gpu):
    return {
        "workload": "C5 metagenome-scale synthetic gene calls (BASELINE.json configs[4]), weak-scaled: "
                    "%d reads x 30 calls per GPU, k=%d, 60k-gene vocabulary, 50 genomes, 1%% false/missing/"
                    "strand-flipped calls; 8 GPUs = the 10M-read set" % (reads_per_gpu, cfg.k),
        "reads_per_gpu": reads_per_gpu, "reads_total": reads_per_gpu * n_gpus, "k": cfg.k, "vocab": cfg.vocab,
        "sharding": "contiguous reads per rank; canonical gene-mers owned by hash range, records routed over NVLink" if n_gpus > 1
                    else "single GPU",
        "l2": "inputs larger than L2 (150 MB of gene ids + ~1 GB of per-build arrays per GPU); no explicit flush",
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.rows, self.proc, self.dev = [], None, device_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-i", str(self.dev), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception as e:          # no nvidia-smi: report it instead of failing the bench
            log("clock sampler unavailable:", e)
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


DUMP_ROWS = 1 << 17
DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """every array as float64 (exact for these integer arrays); one with more than DUMP_ROWS rows is replaced by the
    rows at a fixed seeded sample of indices, which go to <name>_rows.npy, so that the dump stays within DUMP_BYTES"""
    os.makedirs(path, exist_ok=True)
    total = 0
    for name, a in sorted(arrays.items()):
        if not isinstance(a, np.ndarray) or a.ndim == 0:
            continue
        if len(a) > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(len(a), DUMP_ROWS, replace=False)).astype(np.float64)
            np.save(os.path.join(path, name + "_rows.npy"), rows)
            total += rows.nbytes
            a = a[rows.astype(np.int64)]
        a = a.astype(np.float64)
        np.save(os.path.join(path, name + ".npy"), a)
        total += a.nbytes
    assert total <= DUMP_BYTES, total
    log("dumped the last timed build's arrays to %s (%.1f MB)" % (path, total / 2**20))


def pinned(arr):
    import torch
    t = torch.empty(arr.shape, dtype=torch.from_numpy(arr[:0]).dtype, pin_memory=True)
    t.numpy()[...] = arr
    return t


# ------------------------------------------------------------------------------------------------ CPU arms
def time_c_oracle(ids, off, k, n_reads):
    """plain-C restatement (oracle/gmg_oracle.c, 1 thread) on the first n_reads reads -> (gene-mers/s, seconds, W)"""
    from amira_b200 import synth
    from oracle import c_oracle
    o = off[: n_reads + 1]
    i = ids[: int(o[-1])]
    W = synth.count_windows(o, k)
    t = time.perf_counter()
    g = c_oracle.COracleGraph(i, o, k)
    dt = time.perf_counter() - t
    del g
    return W / dt, dt, W


def _big_stack(fn):
    """upstream's component DFS is recursive (construct_graph.py:911-918): run it with a deep stack"""
    out = {}

    def run():
        try:
            out["v"] = fn()
        except BaseException as e:      # noqa: BLE001
            out["e"] = e
    old = sys.getrecursionlimit()
    threading.stack_size(1 << 30)
    sys.setrecursionlimit(10_000_000)
    try:
        t = threading.Thread(target=run)
        t.start()
        t.join()
    finally:
        sys.setrecursionlimit(old)
        threading.stack_size(0)
    if "e" in out:
        raise out["e"]
    return out["v"]


def time_upstream(ids, off, k, n_reads, names, keep=False):
    """upstream's own GeneMerGraph(readDict, k) (unmodified, from baseline/_ref or /root/reference) on the first n_reads
    reads, one core -> (gene-mers/s, seconds, W, (graph, reads) or None)"""
    from amira_b200 import synth
    from oracle import ref_harness
    cg = ref_harness.load()
    o = off[: n_reads + 1]
    i = ids[: int(o[-1])]
    reads = synth.to_read_dict(i, o, names)
    W = synth.count_windows(o, k)
    t = time.perf_counter()
    g = _big_stack(lambda: cg.GeneMerGraph(reads, k))
    dt = time.perf_counter() - t
    return W / dt, dt, W, (g, reads) if keep else None


def upstream_available():
    try:
        from oracle import ref_harness
        return ref_harness.available()
    except Exception:
        return False


def run_reference(args):
    """--impl reference: upstream's own Python implementation of the path on the host CPU.

    `GeneMerGraph(readDict, k)` of the unmodified upstream package (baseline/_ref, installed from /root/reference by
    baseline/install_ref.py; nothing of this repository's engine is on the path), single-process as at every
    upstream call site (cores=1; the result is defined by the sequential dict insertion order).  Upstream builds
    ~10-15k gene-mers/s, so every step is a bounded sample: the first n reads of rank 0's shard, n chosen from a
    pilot run so that warm-up + steps end within ~2.5 minutes.  The plain-C restatement (oracle/gmg_oracle.c) is
    reported beside it as a second, labelled figure."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from amira_b200 import synth
    from oracle import c_oracle
    cfg, ids, off = workload(args.gpus, 0, args.reads_per_gpu)
    k = cfg.k
    base = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic", "config": config_dict(cfg, args.gpus, args.reads_per_gpu), "gpu_launches": 0}
    c_oracle.build()
    n_port = min(args.reads_per_gpu, 400_000)
    port_rate, port_dt, port_w = time_c_oracle(ids, off, k, n_port)
    port = {"value": port_rate, "unit": UNIT, "cores": 1, "kind": "port", "seconds": round(port_dt, 2),
            "sample": "plain-C restatement of the same build (oracle/gmg_oracle.c), first %d reads, %d gene-mers" % (n_port, port_w)}
    if not upstream_available():
        # no upstream package on this box: the C port alone (kind "port")
        t0 = time.perf_counter()
        Wt = 0
        for _ in range(args.steps):
            Wt += time_c_oracle(ids, off, k, n_port)[2]
        dt = time.perf_counter() - t0
        value = Wt / dt
        port["sample"] += " (upstream package not present: baseline/_ref missing)"
        port["value"] = value
        base.update({"value": value, "ms_per_step": dt / args.steps * 1e3, "cpu_baseline": dict(port, host_cores=os.cpu_count()),
                     "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        emit(base)
        return 0
    names = synth.vocabulary_names(cfg.vocab)
    pilot_rate, _, _, _ = time_upstream(ids, off, k, 300, names)
    budget_s = 150.0 / max(1, args.steps + args.warmup)
    per_read = (cfg.fixed_len - k + 1) if cfg.fixed_len else cfg.mean_len
    n = int(min(args.reads_per_gpu, max(300, 0.8 * budget_s * pilot_rate / per_read)))
    for _ in range(args.warmup):
        time_upstream(ids, off, k, n, names)
    t0 = time.perf_counter()
    Wt = 0
    for _ in range(args.steps):
        Wt += time_upstream(ids, off, k, n, names)[2]
    dt = time.perf_counter() - t0
    value = Wt / dt
    sample = ("first %d reads of rank 0's shard (%d gene-mers per step): upstream's unmodified GeneMerGraph(readDict, %d), "
              "CPython %s, 1 of %d host cores" % (n, Wt // max(1, args.steps), k, sys.version.split()[0], os.cpu_count()))
    base.update({
        "value": value, "ms_per_step": dt / args.steps * 1e3,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "reference", "sample": sample,
                         "host_cores": os.cpu_count()},
        "cpu_port": port,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    emit(base)
    return 0


# ------------------------------------------------------------------------------------------------ parity helpers
def load_digests():
    if os.path.exists(DIGESTS):
        with open(DIGESTS) as f:
            return json.load(f)
    return {}


def check_staged(dg, name, ids, off, k, gold, stream):
    """build + rlcc(5) + filter(3,1) on the device, every stage against the oracle's digests -> (ok, times, mismatches)"""
    import torch
    from oracle import digests
    bad, times = [], {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def snap(stage):
        a = dg.arrays()
        want = gold["stages"][stage]
        got_g, got_r = digests.global_digest(a), digests.rank_digest(a)
        for f in digests.diff_digests(got_g, want["global"]) + digests.diff_digests(got_r, want["rank"]):
            bad.append("%s/%s/%s" % (name, stage, f))

    def timed(label, fn):
        dg.sync()
        e0.record(stream)
        fn()
        dg.sync()
        e1.record(stream)
        stream.synchronize()
        times[label] = round(e0.elapsed_time(e1), 4)
    with torch.cuda.stream(stream):
        d_ids, d_off = torch.from_numpy(ids).cuda(), torch.from_numpy(off).cuda()
    stream.synchronize()
    # one untimed cycle first: the handle allocates its filter buffers on first use (Amira reuses one handle for the
    # 10-100 rebuilds of a sample)
    for _ in range(2):
        dg.build(d_ids, d_off, k, on_device=True, wait=False)
    dg.remove_low_coverage_components(5)
    dg.filter_graph(3, 1)
    dg.build(d_ids, d_off, k, on_device=True, wait=False)
    timed("build_ms", lambda: dg.build(d_ids, d_off, k, on_device=True, wait=False))
    snap("build")
    timed("rlcc5_ms", lambda: dg.remove_low_coverage_components(5))
    snap("rlcc5")
    timed("filter3_1_ms", lambda: dg.filter_graph(3, 1))
    snap("rlcc5_filter3_1")
    return not bad, times, bad


# ------------------------------------------------------------------------------------------------ GPU arm
def run_gpu(args):
    import torch
    import torch.distributed as dist

    from amira_b200 import _lib, synth
    from amira_b200.device_graph import DeviceGraph
    from oracle import digests

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        log("WORLD_SIZE %d != --gpus %d; using WORLD_SIZE" % (world, args.gpus))
    n_gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    gloo = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        gloo = dist.new_group(backend="gloo")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg, ids, off = workload(n_gpus, rank, args.reads_per_gpu)
    k = cfg.k
    R = len(off) - 1
    W = synth.count_windows(off, k)
    stream = torch.cuda.Stream()
    dg = DeviceGraph(local_rank, stream=stream.cuda_stream)
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            uid = torch.from_numpy(dg.nccl_unique_id().copy())
        uid = uid.cuda()
        dist.broadcast(uid, 0)
        dg.comm_init(uid.cpu().numpy(), rank, world)

    h_ids, h_off = pinned(ids), pinned(off)
    with torch.cuda.stream(stream):
        d_ids = h_ids.to("cuda", non_blocking=True)
        d_off = h_off.to("cuda", non_blocking=True)
    stream.synchronize()

    # ---- device-resident arm: builds enqueued back to back, no host synchronisation in between -----
    def step_device():
        dg.build(d_ids, d_off, k, on_device=True, wait=False)

    for _ in range(args.warmup):
        step_device()
    dg.sync()
    sizes = dg.sizes()
    launches0 = dg.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        smi_id = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        smi_id = str(local_rank)
    sampler = ClockSampler(smi_id)
    if rank == 0:
        sampler.start()
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    dg.sync()                               # joins the library's side streams into the handle's stream
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = dg.kernel_launches() - launches0
    t = torch.tensor([ms_total], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    w_all = torch.tensor([W], device="cuda", dtype=torch.int64)
    if world > 1:
        dist.all_reduce(w_all)
    W_all = int(w_all.item())
    value = W_all * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dg.arrays())

    # per-phase times and the dominant kernel's duration: CUDA events on the handle's streams, separate untimed builds
    dg.set_profiling(True)
    kern_ms, phase_acc = [], {}
    for _ in range(min(args.steps, 8)):
        dg.build(d_ids, d_off, k, on_device=True, wait=False)
        dg.sync()
        ph = dg.phase_ms()
        kern_ms.append(ph["insert_kernel"])
        for name, ms in ph.items():
            phase_acc[name] = phase_acc.get(name, 0.0) + ms
    dg.set_profiling(False)
    phases = {n: round(v / len(kern_ms), 4) for n, v in phase_acc.items() if v > 0}
    kernel_ms = sum(kern_ms) / len(kern_ms)

    # ---- parity of the timed workload ---------------------------------------------------------------
    gold_all = load_digests()
    parity = {"status": "unchecked"}
    replicated = rank == 0
    dg.build(d_ids, d_off, k, on_device=True)
    mine = dg.arrays(replicated=replicated)
    my_rank_digest = digests.rank_digest(mine)
    gold = gold_all.get("c5_n%d" % n_gpus) if args.reads_per_gpu == READS_PER_GPU else None
    if world > 1:
        pieces = [None] * world
        dist.all_gather_object(pieces, my_rank_digest, group=gloo)
    else:
        pieces = [my_rank_digest]
    if rank == 0:
        bad, against = [], None
        if gold is not None:
            bad += ["global/" + f for f in digests.diff_digests(digests.global_digest(mine), gold["global"])]
            for r, (got, want) in enumerate(zip(pieces, gold["ranks"])):
                bad += ["rank%d/%s" % (r, f) for f in digests.diff_digests(got, want)]
            against = "C oracle digests of the same %d-read workload (tests/golden/bench_digests.json)" % gold["reads"]
        elif n_gpus == 1:
            from oracle import c_oracle
            c_oracle.build()
            ref = c_oracle.COracleGraph(ids, off, k).arrays()
            bad += digests.diff_digests(digests.global_digest(mine), digests.global_digest(ref))
            bad += digests.diff_digests(my_rank_digest, digests.rank_digest(ref))
            against = "C oracle run on the same input in this process"
        if against:
            parity = {"status": "ok" if not bad else "FAIL", "against": against,
                      "fields": len(digests.GLOBAL_FIELDS) + len(digests.RANK_FIELDS) * n_gpus, "mismatches": bad[:20]}
    del mine

    # ---- end-to-end arm: host CSR in, host graph arrays out, through the C ABI ------------------
    # multi-GPU: the node / edge tables are identical on every rank, so rank 0 collects them; every rank
    # exports what it owns (its per-read lists and its share of the node -> read incidence)
    e2e = None
    if not args.no_e2e:
        dg.build(h_ids.numpy(), h_off.numpy(), k)
        out = dg.arrays(replicated=replicated)
        out_pinned = {n: pinned(a).numpy() for n, a in out.items() if isinstance(a, np.ndarray) and a.ndim >= 1 and
                      n not in ("win_start", "win_end")}
        d2h_bytes = int(sum(a.nbytes for a in out_pinned.values()))
        h2d_bytes = int(ids.nbytes + off.nbytes)
        if world > 1:                                 # bytes per step of the whole job
            tb = torch.tensor([h2d_bytes, d2h_bytes], device="cuda", dtype=torch.int64)
            dist.all_reduce(tb)
            h2d_bytes, d2h_bytes = int(tb[0].item()), int(tb[1].item())

        def step_e2e():
            dg.build(h_ids.numpy(), h_off.numpy(), k, wait=False)
            dg.arrays(out=out_pinned, replicated=replicated)

        n_e2e = max(3, min(args.steps, 10))
        for _ in range(2):
            step_e2e()
        barrier()
        e0.record(stream)
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            step_e2e()
        e1.record(stream)
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        e2e_ms = max(e0.elapsed_time(e1), wall_ms)      # exports end with a host sync: wall covers the D2H tail
        t = torch.tensor([e2e_ms], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
        e2e = {"value": W_all * n_e2e / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e_ms / n_e2e, "steps": n_e2e,
               "what": "pinned host CSR -> amira_gmg_build -> amira_gmg_export_{nodes,edges,reads} into pinned host arrays"
                       + (" (every rank: its per-read lists and incidence share; rank 0: also the replicated node / edge "
                          "tables; bytes are the job's total)" if n_gpus > 1 else "")}
    clocks = sampler.stop() if rank == 0 else None   # sampled from the start of the timed region to here

    # ---- roofline of the dominant kernel and of the whole build --------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        with open(peaks_path) as f:
            hbm_peak = float(json.load(f)["hbm_gbs"])
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        hbm_peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    bytes_alg = BYTES_PER_GENE_MER * W + 4 * R * (k - 1) + 8 * R
    achieved = bytes_alg / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "insert_kernel_traffic.json")
    if os.path.exists(tpath) and args.reads_per_gpu == READS_PER_GPU:
        with open(tpath) as f:
            tj = json.load(f)
        traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
    roofline = {"bound": "hbm", "achieved": round(achieved, 2), "peak": hbm_peak, "unit": "GB/s",
                "frac": round(achieved / hbm_peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "k_insert_windows", "kernel_ms": round(kernel_ms, 4), "bytes_per_gene_mer": BYTES_PER_GENE_MER,
                "algorithmic_bytes_per_launch": int(bytes_alg), "peak_source": peak_src,
                "whole_build_frac": round(bytes_alg / (ms_total / args.steps * 1e-3) / 1e9 / hbm_peak, 4)}
    if rank == 0 and not args.no_atomic_peak:
        # the second roofline of SURVEY.md 8(d): algorithmic atomics / measured random-address atomic rate
        red, cas, ld = dg.atomic_peak(64 << 20, 1 << 26)
        t_atomic_ms = ATOMICS_PER_GENE_MER * W / red * 1e3
        roofline["atomic"] = {"red_add_per_s": red, "cas_per_s": cas, "sector_load_per_s": ld,
                              "table": "64 MB (L2 resident)", "atomics_per_gene_mer": ATOMICS_PER_GENE_MER,
                              "kernel_frac": round(t_atomic_ms / kernel_ms, 4),
                              "whole_build_frac": round(t_atomic_ms / (ms_total / args.steps), 4)}

    result = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic", "config": config_dict(cfg, n_gpus, args.reads_per_gpu),
        "graph": {"gene_mers": W_all, "nodes": sizes["nodes"], "edges": sizes["edges"]},
        "parity": parity, "e2e": e2e, "gpu_launches": int(launches), "phases_ms": phases, "roofline": roofline,
        "clocks": clocks, "library": _lib.load().amira_version().decode(),
    }

    # ---- CPU baseline beside it (rank 0, N=1 only) ----------------------------------------------
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        from oracle import c_oracle
        from oracle import gmg_oracle as O
        c_oracle.build()
        port_rate, port_dt, port_w = time_c_oracle(ids, off, k, min(R, args.cpu_sample_reads))
        port = {"value": port_rate, "unit": UNIT, "cores": 1, "kind": "port", "seconds": round(port_dt, 2),
                "sample": "plain-C restatement of upstream's single-process build (oracle/gmg_oracle.c), first %d of the %d "
                          "reads of the same workload, %d gene-mers" % (min(R, args.cpu_sample_reads), R, port_w)}
        if upstream_available():
            names = synth.vocabulary_names(cfg.vocab)
            pilot, _, _, _ = time_upstream(ids, off, k, 300, names)
            per_read = (cfg.fixed_len - k + 1) if cfg.fixed_len else cfg.mean_len
            n = int(min(R, max(300, args.cpu_seconds * pilot / per_read)))
            rate, dt, w, keep = time_upstream(ids, off, k, n, names, keep=True)
            # the same sample through the GPU path, against upstream's own objects (not only against the restatement)
            from oracle import ref_harness
            up_graph, up_reads = keep
            up = ref_harness.reference_arrays(up_graph, list(up_reads), names)
            o_s = off[: n + 1]
            dg.build(ids[: int(o_s[-1])], o_s, k)
            d = O.diff_arrays(dg.arrays(), up, [f for f in O.ARRAY_FIELDS if f not in ("win_start", "win_end")])
            result["cpu_baseline"] = {
                "value": rate, "unit": UNIT, "cores": 1, "kind": "reference", "host_cores": os.cpu_count(), "seconds": round(dt, 2),
                "sample": "first %d of the %d reads of the same workload (%d gene-mers): upstream's unmodified "
                          "GeneMerGraph(readDict, %d) from baseline/_ref, CPython %s, 1 core (upstream's build is "
                          "single-process at every call site)" % (n, R, w, k, sys.version.split()[0]),
                "parity_vs_upstream": "ok" if not d else "FAIL %r" % (d,)}
            result["cpu_port"] = port
            if d and result["parity"].get("status") != "FAIL":
                result["parity"] = {"status": "FAIL", "against": "upstream GeneMerGraph on the CPU sample", "mismatches": d}
        else:
            result["cpu_baseline"] = port

    # ---- the other BASELINE.json configs on one GPU (extra keys, not the headline) -----------------
    if rank == 0 and n_gpus == 1 and not args.no_extras:
        extras, bad_all = {}, []
        # C2: 50k reads, k=3: small-graph regime, the repeated build is replayed as one CUDA graph
        c2 = synth.CONFIGS["c2"]
        i2, o2 = synth.generate(c2, 0, c2.n_reads)
        w2 = synth.count_windows(o2, c2.k)
        with torch.cuda.stream(stream):
            di, do = torch.from_numpy(i2).cuda(), torch.from_numpy(o2).cuda()
        stream.synchronize()
        for _ in range(6):
            dg.build(di, do, c2.k, on_device=True, wait=False)
        dg.sync()
        g0 = dg.kernel_launches()
        e0.record(stream)
        for _ in range(50):
            dg.build(di, do, c2.k, on_device=True, wait=False)
        dg.sync()
        e1.record(stream)
        stream.synchronize()
        ms2 = e0.elapsed_time(e1) / 50
        extras["c2_isolate"] = {"workload": "BASELINE.json configs[1]: 50k reads x ~25 calls, 6k vocab, k=3", "gene_mers": w2,
                                "ms_per_graph": round(ms2, 4), "gene_mers_per_s": w2 / (ms2 * 1e-3),
                                "kernels_per_graph": (dg.kernel_launches() - g0) // 50,
                                "launch": "one cudaGraphLaunch per build (captured on the second repeat of the same input)"}
        if "c2_k3" in gold_all:
            ok, tm, bad = check_staged(dg, "c2_k3", i2, o2, 3, gold_all["c2_k3"], stream)
            extras["c2_isolate"].update({"parity": "ok" if ok else "FAIL", "stages_ms": tm})
            bad_all += bad
        # C3: 500k reads, 10% bad calls, k = 3 / 5 / 7, then remove_low_coverage_components(5) + filter_graph(3, 1)
        c3 = synth.CONFIGS["c3"]
        i3, o3 = synth.generate(c3, 0, c3.n_reads)
        extras["c3_high_error"] = {"workload": "BASELINE.json configs[2]: 500k reads, 10% false/missing/strand-flipped calls"}
        for kk in (3, 5, 7):
            key = "c3_k%d" % kk
            if key not in gold_all:
                continue
            ok, tm, bad = check_staged(dg, key, i3, o3, kk, gold_all[key], stream)
            w3 = synth.count_windows(o3, kk)
            tm.update({"gene_mers": w3, "gene_mers_per_s": w3 / (tm["build_ms"] * 1e-3), "parity": "ok" if ok else "FAIL"})
            extras["c3_high_error"]["k%d" % kk] = tm
            bad_all += bad
        del i3, o3
        # C4: 2M reads, 12 genomes, 60k vocabulary, k=3 -- the whole set on one GPU
        if "c4_k3" in gold_all and not args.no_c4:
            c4 = synth.CONFIGS["c4"]
            i4, o4 = synth.generate(c4, 0, c4.n_reads)
            ok, tm, bad = check_staged(dg, "c4_k3", i4, o4, 3, gold_all["c4_k3"], stream)
            w4 = synth.count_windows(o4, 3)
            tm.update({"workload": "BASELINE.json configs[3]: 2M reads, 12 genomes, 60k vocabulary, k=3 (one GPU)",
                       "gene_mers": w4, "gene_mers_per_s": w4 / (tm["build_ms"] * 1e-3), "parity": "ok" if ok else "FAIL"})
            extras["c4_multi_genome"] = tm
            bad_all += bad
        # the drop-in PYTHON class (what Amira itself calls): read dict in -> graph object -> first accessors out.
        # Host-side string encoding and the lazily materialised views are inside the time; best of 3.
        try:
            from amira_b200 import GeneMerGraph
            py = {}
            for tag, cfg, n_r in (("config1_scale", synth.CONFIGS["c2"], 21000), ("c2_isolate", synth.CONFIGS["c2"], c2.n_reads)):
                ii, oo = synth.generate(cfg, 0, n_r)
                rd = synth.to_read_dict(ii, oo, synth.vocabulary_names(cfg.vocab))
                best = None
                for _ in range(3):
                    t0 = time.perf_counter()
                    gg = GeneMerGraph(rd, 3)
                    nn, ne = gg.get_total_number_of_nodes(), gg.get_total_number_of_edges()
                    t1 = time.perf_counter()
                    mean_cov = gg.get_mean_node_coverage()
                    first = next(iter(gg.all_nodes()))
                    cov0 = first.get_node_coverage()
                    t2 = time.perf_counter()
                    cur = ((t1 - t0) * 1e3, (t2 - t0) * 1e3)
                    best = cur if best is None or cur[1] < best[1] else best
                py[tag] = {"reads": n_r, "gene_mers": synth.count_windows(oo, 3), "nodes": nn, "edges": ne,
                           "constructor_and_counts_ms": round(best[0], 2), "plus_mean_coverage_and_first_node_ms": round(best[1], 2)}
                del gg, rd
            py["what"] = ("GeneMerGraph(readDict, 3) of the drop-in class on string gene calls (synthetic C2 generator; config1_scale = "
                          "the read count of tests/complex_gene_calls_one.json, which does not travel to the GPU box): encode + "
                          "device build + node/edge counts, then mean node coverage and the first Node object")
            extras["python_class"] = py
        except Exception as exc:  # the headline does not depend on it
            extras["python_class"] = {"error": repr(exc)}
        if bad_all:
            result["parity"] = {"status": "FAIL", "against": "C oracle digests of the extra configs", "mismatches": bad_all[:20]}
        result["extras"] = extras
        result["c2_isolate"] = extras["c2_isolate"]
    rc = 0
    if rank == 0:
        emit(result)
        if result["parity"].get("status") == "FAIL":
            log("PARITY FAILURE:", result["parity"])
            rc = 3
    dg.close()
    if world > 1:
        dist.destroy_process_group()
    return rc


def main():
    # NCCL and friends print banners on stdout; the contract is ONE JSON line there, so everything else
    # (including native code writing to fd 1) is sent to stderr and the line goes to the saved descriptor
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads-per-gpu", type=int, default=READS_PER_GPU)
    ap.add_argument("--cpu-sample-reads", type=int, default=READS_PER_GPU, help="reads of the C-port figure")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU time budget of the upstream sample in the GPU arm")
    ap.add_argument("--phases", action="store_true", help="(kept for compatibility; phase times are always reported)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-atomic-peak", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C2 / C3 / C4 extra configs")
    ap.add_argument("--no-c2", action="store_true", help="alias of --no-extras")
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end arm (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays of the last timed build to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.no_extras = args.no_extras or args.no_c2
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
