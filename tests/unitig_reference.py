"""Reference for amira_gmg_unitigs: a plain loop that restates its definition (include/amira_gmg.h) over the exported
arrays, and the oracle-backed test double with DeviceGraph.unitigs built on it.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

from tests.fake_device import OracleBackedDevice


def unitig_succ(a):
    """succ of every state 2 * node + side, one at a time: list `side` of u holds exactly one edge (u -> v, td),
    v != u, and v's entering list (backward if td == +1, forward if td == -1) holds exactly one edge"""
    fw_off, fw_edges, bw_off, bw_edges = (a[f].tolist() for f in ("fw_off", "fw_edges", "bw_off", "bw_edges"))
    tgt, td = a["edge_tgt"].tolist(), a["edge_td"].tolist()

    def lst(n, side):
        return fw_edges[fw_off[n]:fw_off[n + 1]] if side == 0 else bw_edges[bw_off[n]:bw_off[n + 1]]

    out = []
    for s in range(2 * len(a["node_cov"])):
        u, side = s >> 1, s & 1
        e = lst(u, side)
        if len(e) != 1:
            out.append(-1)
            continue
        v, leave = tgt[e[0]], 0 if td[e[0]] == 1 else 1
        out.append(2 * v + leave if v != u and len(lst(v, 1 - leave)) == 1 else -1)
    return out


def unitig_loop(a):
    """the unitigs of the graph arrays `a`, walked state by state -> the dict DeviceGraph.unitigs returns"""
    N = len(a["node_cov"])
    nxt = unitig_succ(a)
    prv = [-1] * (2 * N)
    for s, t in enumerate(nxt):
        if t >= 0:
            assert prv[t] == -1, "two predecessors of state %d" % t
            prv[t] = s
    cov = a["node_cov"].tolist()
    node_unitig, node_pos, node_orient = [-1] * N, [0] * N, [0] * N
    off, order, circular, cov_sum, cov_min, cov_max = [0], [], [], [], [], []
    for m in range(N):                                  # the first node not yet seen is its unitig's smallest
        if node_unitig[m] >= 0:
            continue
        head, circ = 2 * m, False
        while prv[head] >= 0:
            head = prv[head]
            if head == 2 * m:
                circ = True
                break
        chain, t = [head], nxt[head]
        while t >= 0 and t != head:
            chain.append(t)
            t = nxt[t]
        u = len(circular)
        for p, s in enumerate(chain):
            n = s >> 1
            assert node_unitig[n] == -1, "node %d in two unitigs" % n
            node_unitig[n], node_pos[n], node_orient[n] = u, p, -1 if s & 1 else 1
            order.append(n)
        off.append(len(order))
        circular.append(int(circ))
        c = [cov[s >> 1] for s in chain]
        cov_sum.append(sum(c))
        cov_min.append(min(c))
        cov_max.append(max(c))
    # the edge of every link s -> succ(s): the one edge of list s & 1 of node s >> 1
    fw_off, fw_edges, bw_off, bw_edges = (a[f].tolist() for f in ("fw_off", "fw_edges", "bw_off", "bw_edges"))
    internal = [0] * len(a["edge_src"])
    for s, t in enumerate(nxt):
        if t >= 0:
            internal[fw_edges[fw_off[s >> 1]] if s & 1 == 0 else bw_edges[bw_off[s >> 1]]] = 1
    return {"node_unitig": np.asarray(node_unitig, np.int32), "node_pos": np.asarray(node_pos, np.int32),
            "node_orient": np.asarray(node_orient, np.int8), "unitig_off": np.asarray(off, np.int64),
            "unitig_nodes": np.asarray(order, np.int32), "circular": np.asarray(circular, np.uint8),
            "cov_sum": np.asarray(cov_sum, np.int64), "cov_min": np.asarray(cov_min, np.uint32),
            "cov_max": np.asarray(cov_max, np.uint32), "edge_internal": np.asarray(internal, np.uint8)}


class UnitigDevice(OracleBackedDevice):
    """the test double with unitigs: unitig_loop over the oracle's arrays, as DeviceGraph.unitigs"""

    def unitigs(self):
        return unitig_loop(self.arrays())
