"""Reference for amira_gmg_unitig_links and amira_gmg_read_unitig_paths: plain loops that restate their definitions
(include/amira_gmg.h) over the exported arrays `a` and unitig_loop's output `u`, and the test double with
DeviceGraph.unitig_links / read_unitig_paths built on them.  read_path_loop uses the position form of the definition
(one unitig, one orientation, the position moving by one in the direction of travel), not succ, so that it and the
library come from two formulations.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

from tests.unitig_reference import UnitigDevice, unitig_loop


def link_loop(a, u):
    """one link per junction edge (edge_internal == 0), in edge order"""
    out = {f: [] for f in ("edge", "from_unitig", "from_orient", "to_unitig", "to_orient", "cov")}
    src, tgt, sd, td = (a[f].tolist() for f in ("edge_src", "edge_tgt", "edge_sd", "edge_td"))
    cov, internal = a["edge_cov"].tolist(), u["edge_internal"].tolist()
    nu, no = u["node_unitig"].tolist(), u["node_orient"].tolist()
    for j in range(len(src)):
        if internal[j]:
            continue
        out["edge"].append(j)
        out["from_unitig"].append(nu[src[j]])
        out["from_orient"].append(sd[j] * no[src[j]])
        out["to_unitig"].append(nu[tgt[j]])
        out["to_orient"].append(td[j] * no[tgt[j]])
        out["cov"].append(cov[j])
    return {"edge": np.asarray(out["edge"], np.int32), "from_unitig": np.asarray(out["from_unitig"], np.int32),
            "from_orient": np.asarray(out["from_orient"], np.int8), "to_unitig": np.asarray(out["to_unitig"], np.int32),
            "to_orient": np.asarray(out["to_orient"], np.int8), "cov": np.asarray(out["cov"], np.uint32)}


def read_path_loop(a, u):
    """per read, window by window: a live window extends the current step when it lies on the same unitig with the
    same orientation, one position further in the direction of travel (modulo a circular unitig's length)"""
    woff, wn, wd = a["win_off"].tolist(), a["win_node"].tolist(), a["win_dir"].tolist()
    nu, npos, no = u["node_unitig"].tolist(), u["node_pos"].tolist(), u["node_orient"].tolist()
    ulen, circ = np.diff(u["unitig_off"]).tolist(), u["circular"].tolist()
    path_off, steps = [0], []               # steps: [unitig, orient, pos, win, length, position of the last window]
    for r in range(len(woff) - 1):
        cur = None
        for i in range(woff[r + 1] - woff[r]):
            n = wn[woff[r] + i]
            if n < 0:
                cur = None
                continue
            un, o, p = nu[n], wd[woff[r] + i] * no[n], npos[n]
            if cur is not None and cur[0] == un and cur[1] == o:
                nxt = cur[5] + o
                if circ[un]:
                    nxt %= ulen[un]
                if p == nxt:
                    cur[4] += 1
                    cur[5] = p
                    continue
            cur = [un, o, p, i, 1, p]
            steps.append(cur)
        path_off.append(len(steps))
    col = list(zip(*steps)) if steps else [[]] * 6
    return {"path_off": np.asarray(path_off, np.int64), "unitig": np.asarray(col[0], np.int32),
            "orient": np.asarray(col[1], np.int8), "pos": np.asarray(col[2], np.int32), "win": np.asarray(col[3], np.int32),
            "length": np.asarray(col[4], np.int32)}


class UnitigPathDevice(UnitigDevice):
    """the test double with unitig_links and read_unitig_paths: the loops over the oracle's arrays"""

    def unitig_links(self):
        a = self.arrays()
        return link_loop(a, unitig_loop(a))

    def read_unitig_paths(self):
        a = self.arrays()
        return read_path_loop(a, unitig_loop(a))
