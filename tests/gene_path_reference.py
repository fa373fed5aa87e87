"""amira_gmg_gene_paths restated as plain loops over its definition (include/amira_gmg.h): occurrences walked window by
window, clusters in a dict keyed by tuples, and a partial occurrence tested against every key at every position.  The
CPU and GPU tests compare the product's numpy implementation and the device with it."""
import numpy as np


def marked_nodes(a, ranks):
    """marked[n]: node n's gene-mer holds one of the genes (by rank, either strand)"""
    key = np.asarray(a["node_key"])
    return [any(abs(int(x)) in set(ranks) for x in row) for row in key.tolist()]


def gene_path_loop(w, marked) -> dict:
    """the outputs of amira_gmg_gene_paths for the windows w (win_off, win_node with -1 for None, win_dir) and the
    marked nodes"""
    woff = [int(x) for x in w["win_off"]]
    node = [int(x) for x in w["win_node"]]
    dirs = [int(x) for x in w["win_dir"]]
    occ = []                                    # (read, first window, length, left flank, right flank, span)
    for r in range(len(woff) - 1):
        lo, hi = woff[r], woff[r + 1]
        nw = hi - lo
        i = 0
        while i < nw:
            n = node[lo + i]
            if n < 0 or not marked[n]:
                i += 1
                continue
            j = i
            while j + 1 < nw and node[lo + j + 1] >= 0 and marked[node[lo + j + 1]]:
                j += 1
            left = i >= 1 and node[lo + i - 1] >= 0
            right = j + 1 < nw and node[lo + j + 1] >= 0
            a, b = i - 1 if left else i, j + 1 if right else j
            span = tuple(2 * node[lo + x] + (1 if dirs[lo + x] < 0 else 0) for x in range(a, b + 1))
            occ.append((r, i, j - i + 1, left, right, span))
            i = j + 1
    clusters = {}
    cluster, orient = [], []
    for r, i, ln, left, right, S in occ:
        RS = tuple(s ^ 1 for s in reversed(S))
        orient.append(1 if S <= RS else -1)
        if left and right:
            cluster.append(clusters.setdefault(min(S, RS), len(clusters)))
        else:
            cluster.append(None)
    keys = list(clusters)

    def contains(key, x):
        return any(key[p:p + len(x)] == x for p in range(len(key) - len(x) + 1))

    for o, (r, i, ln, left, right, S) in enumerate(occ):
        if cluster[o] is not None:
            continue
        RS = tuple(s ^ 1 for s in reversed(S))
        hits = [c for c, key in enumerate(keys) if contains(key, S) or contains(key, RS)]
        if len(hits) == 1:
            cluster[o] = hits[0]
            orient[o] = 1 if contains(keys[hits[0]], S) else -1
        else:
            cluster[o] = -1 if not hits else -2
    members = [[o for o in range(len(occ)) if cluster[o] == c] for c in range(len(keys))]
    complete = [sum(1 for o in m if occ[o][3] and occ[o][4]) for m in members]
    key_off, member_off = [0], [0]
    for c in range(len(keys)):
        key_off.append(key_off[-1] + len(keys[c]))
        member_off.append(member_off[-1] + len(members[c]))
    return {"occ_read": np.asarray([x[0] for x in occ], np.int32), "occ_win": np.asarray([x[1] for x in occ], np.int32),
            "occ_length": np.asarray([x[2] for x in occ], np.int32),
            "occ_flanks": np.asarray([(1 if x[3] else 0) | (2 if x[4] else 0) for x in occ], np.uint8),
            "occ_orient": np.asarray(orient, np.int8), "occ_cluster": np.asarray(cluster, np.int32),
            "key_off": np.asarray(key_off, np.int64), "key_state": np.asarray([s for k in keys for s in k], np.int32),
            "n_complete": np.asarray(complete, np.uint32), "member_off": np.asarray(member_off, np.int64),
            "members": np.asarray([o for m in members for o in m], np.int32)}


GENE_PATH_FIELDS = ("occ_read", "occ_win", "occ_length", "occ_flanks", "occ_orient", "occ_cluster", "key_off",
                    "key_state", "n_complete", "member_off", "members")


def same_gene_paths(x, y, ctx=""):
    for f in GENE_PATH_FIELDS:
        assert x[f].dtype == y[f].dtype, (ctx, f, x[f].dtype, y[f].dtype)
        assert np.array_equal(x[f], y[f]), (ctx, f, x[f][:20], y[f][:20])
