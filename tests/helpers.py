"""shared test helpers: golden input loading, stage application, digests of post-build scan results"""
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
POSTBUILD = os.path.join(GOLD, "postbuild.json")

with open(os.path.join(GOLD, "expected.json")) as _f:
    EXPECTED = json.load(_f)
GOLDEN_KEYS = sorted(k for k in EXPECTED if not k.startswith("_"))
STAGE_ORDER = ("build", "rlcc5", "rlcc5_filter3_1")


def load_input(name):
    z = np.load(os.path.join(GOLD, "inputs", name + ".npz"))
    ids = z["ids"].astype(np.int32)
    off = z["off"].astype(np.int64)
    ps = z["pos_start"].astype(np.int32) if "pos_start" in z.files else None
    pe = z["pos_end"].astype(np.int32) if "pos_end" in z.files else None
    return [str(x) for x in z["vocab"]], ids, off, ps, pe


def apply_stage(graph, stage):
    """graph: anything with remove_low_coverage_components / filter_graph"""
    if stage == "rlcc5":
        graph.remove_low_coverage_components(5)
    elif stage == "rlcc5_filter3_1":
        graph.filter_graph(3, 1)


def read_dict(vocab, ids, off, ps=None, pe=None):
    toks = [("+" if x > 0 else "-") + vocab[abs(int(x)) - 1] for x in ids.tolist()]
    reads = {"read%09d" % i: toks[off[i]:off[i + 1]] for i in range(len(off) - 1)}
    pos = None
    if ps is not None:
        pos = {r: [[int(ps[j]), int(pe[j])] for j in range(off[i], off[i + 1])] for i, r in enumerate(reads)}
    return reads, pos


def _canon(v):
    """JSON form under which two results are equal when Python's == says so: sets sorted, graph objects by hash;
    int and float stay apart, so a digest also checks the types of coverage statistics"""
    if isinstance(v, dict):
        return {str(k): _canon(x) for k, x in v.items()}
    if isinstance(v, (set, frozenset)):
        return sorted((_canon(x) for x in v), key=json.dumps)
    if isinstance(v, (list, tuple)):
        return [_canon(x) for x in v]
    if isinstance(v, np.generic):
        return v.item()
    if v is None or isinstance(v, (str, int, float)):
        return v
    return hex(v.__hash__())


def digest(value):
    return hashlib.sha256(json.dumps(_canon(value), sort_keys=True).encode()).hexdigest()


def check_postbuild(key, values):
    """`values` (label -> result) against the digests stored under `key` in tests/golden/postbuild.json"""
    with open(POSTBUILD) as f:
        want = json.load(f)[key]
    got = {label: digest(v) for label, v in values.items()}
    assert got.keys() == want.keys(), (key, sorted(got.keys() ^ want.keys()))
    assert got == want, (key, [label for label in want if got[label] != want[label]])
