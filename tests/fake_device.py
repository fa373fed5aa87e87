"""Test double for amira_b200.device_graph.DeviceGraph backed by the C oracle, so that the host-side
mirror (encoding, materialisation, removal mirroring, upstream binding) can be exercised on a box
without a GPU, and so that the GPU tests have a reference for every post-build scan and edit.
TEST INFRASTRUCTURE ONLY -- the product never uses it."""
import numpy as np

from oracle import c_oracle


class OracleBackedDevice:
    def __init__(self, device=0):
        self.owner = None
        self._g = None
        self._masks = None

    def build(self, ids, off, k, pos_start=None, pos_end=None, on_device=False):
        self._g = c_oracle.COracleGraph(ids, off, k, pos_start, pos_end)
        self.k, self.R, self.has_pos = k, len(off) - 1, pos_start is not None
        self._read_len = np.diff(np.asarray(off, np.int64))
        self._masks = None
        return self

    def build_resident(self, encoded, k, device=None):
        return self.build(encoded.ids, encoded.off, k, encoded.pos_start, encoded.pos_end)

    # ---- the post-build scans of the C ABI, restated with numpy on the oracle's arrays ----
    def sizes_early(self):
        a = self._g.arrays()
        return {"nodes": len(a["node_cov"]), "edges": len(a["edge_cov"]), "windows": len(a["win_node"]),
                "short_reads": int(a["is_short"].sum())}

    def read_length_coverages(self, min_lens):
        a = self._g.arrays()
        lens = self._read_len[a["node_reads"]]
        return np.asarray([int(np.count_nonzero(lens >= k)) for k in min_lens], np.int64)

    def node_coverage_stats(self):
        c = self._g.arrays()["node_cov"]
        return int(c.sum(dtype=np.int64)), int(c.max()) if len(c) else 0

    def junk_read_mask(self, error_rate):
        """upstream: a read is kept when count(None) <= round(len(nodes) * (1 - error_rate)); np.rint on the same
        float64 product is Python's round-half-even"""
        a = self._g.arrays()
        none = np.concatenate([[0], np.cumsum(a["win_node"] < 0, dtype=np.int64)])
        woff = a["win_off"]
        n_none = none[woff[1:]] - none[woff[:-1]]
        n_win = np.diff(woff).astype(np.float64)
        out = (n_none <= np.rint(n_win * (1 - error_rate))).astype(np.uint8)
        out[a["is_short"] != 0] = 2
        return out

    def nodes_containing(self, ranks):
        key = np.abs(self._g.arrays()["node_key"])
        return np.isin(key, np.asarray(ranks)).any(axis=1) if len(key) else np.zeros(0, bool)

    def linear_steps(self):
        """degree, and per side the step of get_forward_node_from_node (the ONLY forward edge) /
        get_backward_node_from_node (the FIRST backward edge); the walk continues into a target of degree 1 or 2
        that is not the node itself"""
        a = self._g.arrays()
        n = len(a["node_cov"])
        deg = (np.diff(a["fw_off"]) + np.diff(a["bw_off"])).astype(np.uint32)
        out = {"degree": deg}
        for side, off, edges in (("fw", a["fw_off"], a["fw_edges"]), ("bw", a["bw_off"], a["bw_edges"])):
            nxt, dr, ext = np.full(n, -1, np.int32), np.zeros(n, np.int8), np.zeros(n, np.uint8)
            cnt = np.diff(off)
            take = np.flatnonzero(cnt == 1 if side == "fw" else cnt > 0)
            e = edges[off[take]]
            t = a["edge_tgt"][e]
            nxt[take], dr[take] = t, a["edge_td"][e]
            ext[take] = ((deg[t] == 1) | (deg[t] == 2)) & (t != take)
            out[side + "_next"], out[side + "_dir"], out[side + "_ext"] = nxt, dr, ext
        self._masks = None                # the library computes the steps in the memory of the filter masks
        return out

    def arrays(self):
        return self._g.arrays()

    def arrays_reads_only(self):
        return {"win_node": self._g.arrays()["win_node"]}

    def sizes(self):
        a = self._g.arrays()
        return {"nodes": len(a["node_cov"]), "edges": len(a["edge_cov"]), "windows": len(a["win_node"])}

    # ---- edits; filter_masks() describes the last one ----
    def _with_masks(self, op):
        """run `op` on the oracle and derive the keep flags from the arrays before and after it: every node lies on
        a window, so the surviving windows map new node indices to old ones"""
        before = self._g.arrays()
        self._masks = None
        op()
        after = self._g.arrays()
        n = len(before["node_cov"])
        on = after["win_node"] >= 0
        old_idx = np.zeros(len(after["node_cov"]), np.int64)
        old_idx[after["win_node"][on]] = before["win_node"][on]
        assert np.array_equal(before["node_key"][old_idx], after["node_key"]) and np.all(np.diff(old_idx) > 0)
        nk = np.zeros(n, bool)
        nk[old_idx] = True

        def code(a, remap):
            return (remap[a["edge_src"]] * n + remap[a["edge_tgt"]]) * 2 + (a["edge_sd"] * a["edge_td"] > 0)

        old_code = code(before, np.arange(n, dtype=np.int64))
        new_code = code(after, old_idx)
        ek = np.isin(old_code, new_code)
        assert np.array_equal(old_code[ek], new_code)
        self._masks = (nk, ek)

    def filter_graph(self, a, b):
        self._with_masks(lambda: self._g.filter_graph(a, b))
        return self

    def remove_low_coverage_components(self, c):
        self._with_masks(lambda: self._g.remove_low_coverage_components(c))

    def remove_nodes(self, remove_flags):
        f = np.ascontiguousarray(remove_flags, np.uint8)
        assert len(f) == self.sizes_early()["nodes"]
        self._with_masks(lambda: self._g.remove_nodes(f))

    def remove_nodes_without_reads_of(self, ranks):
        """remove_non_AMR_associated_nodes: the reads of the nodes holding one of the genes; every node on none of
        those reads goes"""
        a = self._g.arrays()
        hit = self.nodes_containing(ranks)
        roff, reads = a["node_reads_off"], a["node_reads"]
        node_of = np.repeat(np.arange(len(hit)), np.diff(roff))
        marked = np.zeros(self.R, bool)
        marked[reads[hit[node_of]]] = True
        touches = np.zeros(len(hit), bool)
        touches[node_of[marked[reads]]] = True
        self.remove_nodes(~touches)

    def filter_masks(self):
        if self._masks is None:
            raise RuntimeError("no filter has run on this graph")
        return self._masks
