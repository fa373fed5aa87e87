"""CPU oracle for Amira's gene-space de Bruijn graph build -- TEST INFRASTRUCTURE ONLY.

This module is the *checker*, never the product: only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import it.  Nothing under ``amira_b200/`` imports it.

It is a sequential, dictionary-based restatement of the reference algorithm
(citations are to files under the upstream checkout, ``amira/...``):

* gene token parsing and the signed SHA-256 gene hash  construct_gene.py:5-10, 48-67, 91-93
* reverse complement / canonical choice / direction     construct_gene_mer.py:4-39, 60-70
* node key = SHA-256(pickle(tuple(canonical hashes)))   construct_gene_mer.py:94-97
* window enumeration + window positions                 construct_read.py:37-59
* the build loop, add_node / add_edge / add_node_to_read construct_graph.py:45-100, 165-178, 196-212, 246-324
* edge identity (invariant under flipping both signs)    construct_edge.py:104-124
* component numbering                                   construct_graph.py:911-927
* filter_graph, remove_node, remove_edge                construct_graph.py:409-540
* remove_low_coverage_components                        construct_graph.py:929-958

Parity status: PINNED.  ``oracle/make_golden.py`` runs the unmodified upstream
``GeneMerGraph`` (imported from the read-only checkout in the build container) on the
upstream test fixtures and on seeded synthetic inputs, and commits digests + full dumps
under ``tests/golden/``; ``tests/test_oracle_golden.py`` checks this module against
every one of them.

The result is exposed as *graph arrays* (see ``GraphArrays`` in DESIGN.md): hash-value
independent, keyed by signed SHA-rank gene ids, in the reference's insertion orders.
"""
from __future__ import annotations

import copy
import hashlib
import pickle

import numpy as np


def sha_int(value) -> int:
    """int(sha256(pickle.dumps(value)).hexdigest(), 16)   (construct_gene.py:5-10)"""
    return int.from_bytes(hashlib.sha256(pickle.dumps(value)).digest(), "big")


def parse_call(token: str):
    """'+name' / '-name' -> (name with spaces as underscores, +1 | -1)   (construct_gene.py:49-65)"""
    assert token.replace(" ", "") != "", "Gene information is missing"
    strand_char = token[0]
    name = token[1:].replace(" ", "_")
    assert strand_char == "-" or strand_char == "+", "Strand information missing for: " + token
    assert name != "", "Gene name information missing for: " + token
    return name, (1 if strand_char == "+" else -1)


class _NodeRec:
    __slots__ = ("key", "names", "hash", "cov", "reads", "fw", "bw", "first_dir", "comp")

    def __init__(self, key, names, node_hash, first_dir):
        self.key = key            # tuple of signed gene hashes of the canonical gene-mer
        self.names = names        # tuple of (name, strand) of the canonical gene-mer
        self.hash = node_hash
        self.cov = 0
        self.reads = []           # read ids, first-touch order, unique
        self.fw = []              # edge hashes whose stored source direction is +1
        self.bw = []              # edge hashes whose stored source direction is -1
        self.first_dir = first_dir
        self.comp = None


class _EdgeRec:
    __slots__ = ("hash", "src", "tgt", "sd", "td", "cov")

    def __init__(self, edge_hash, src, tgt, sd, td):
        self.hash, self.src, self.tgt, self.sd, self.td = edge_hash, src, tgt, sd, td
        self.cov = 0


class OracleGraph:
    """Sequential restatement of ``GeneMerGraph.__init__`` + filters on plain records."""

    def __init__(self, reads, k, positions=None):
        self.k = k
        self.reads_in = reads
        self.read_ids = list(reads)
        self.nodes = {}            # node hash -> _NodeRec, insertion ordered
        self.edges = {}            # edge hash -> _EdgeRec, insertion ordered
        self.read_nodes = {}       # rid -> [node hash | None]
        self.read_dirs = {}        # rid -> [+1/-1 | None]
        self.read_pos = {}         # rid -> [(start, end) | None]
        self.short_reads = {}
        self.to_correct = set()
        self.min_node_cov = 1
        self.min_edge_cov = 1
        self.n_windows = 0
        self._gene_hash = {}
        self._node_hash = {}
        self._edge_hash = {}
        for rid in reads:
            pos = positions[rid] if positions else None
            self._add_read(rid, reads[rid], pos)
        self._label_components()

    # ---- primitives -------------------------------------------------------------
    def _signed_hash(self, name, strand):
        h = self._gene_hash.get(name)
        if h is None:
            h = self._gene_hash[name] = sha_int(name)
        return h * strand

    def _window(self, genes, signed, i):
        """canonical key, canonical (name,strand) tuple, direction of window i"""
        k = self.k
        fwd = signed[i:i + k]
        rc = [-x for x in reversed(fwd)]
        assert fwd != rc, "Gene-mer and reverse complement gene-mer are identical"
        if min(fwd, rc) == fwd:           # Python list order == the reference's sorted([...])[0]
            return tuple(fwd), tuple(genes[i:i + k]), 1
        return tuple(rc), tuple((n, -s) for n, s in reversed(genes[i:i + k])), -1

    def _node(self, key, names, direction, rid):
        nh = self._node_hash.get(key)
        if nh is None:
            nh = self._node_hash[key] = sha_int(key)
        rec = self.nodes.get(nh)
        if rec is None:
            rec = self.nodes[nh] = _NodeRec(key, names, nh, direction)
        if rid is not None and rid not in rec.reads:
            rec.reads.append(rid)
        return rec

    def _edge_key(self, a, b):
        """min(SHA((a, b)), SHA((-a, -b))) -- construct_edge.py:104-124"""
        eh = self._edge_hash.get((a, b))
        if eh is None:
            eh = min(sha_int((a, b)), sha_int((-a, -b)))
            self._edge_hash[(a, b)] = self._edge_hash[(-a, -b)] = eh
        return eh

    def _stored_edge(self, src, tgt, sd, td):
        eh = self._edge_key(src.hash * sd, tgt.hash * td)
        rec = self.edges.get(eh)
        if rec is None:
            rec = self.edges[eh] = _EdgeRec(eh, src, tgt, sd, td)
        return rec

    @staticmethod
    def _attach(node, edge):
        lst = node.fw if edge.sd == 1 else node.bw
        if edge.hash not in lst:
            lst.append(edge.hash)

    # ---- build ------------------------------------------------------------------
    def _add_read(self, rid, calls, pos):
        k = self.k
        genes = [parse_call(c) for c in calls]
        n_win = len(genes) - (k - 1) if len(genes) > k - 1 else 0
        if n_win == 0:
            self.short_reads[rid] = calls
            return
        assert k >= 1, "Gene-mer is empty"
        signed = [self._signed_hash(n, s) for n, s in genes]
        wins = [self._window(genes, signed, i) for i in range(n_win)]
        wpos = [((pos[i][0], pos[i + k - 1][1]) if pos else None) for i in range(n_win)]
        self.n_windows += n_win
        self.read_nodes[rid], self.read_dirs[rid], self.read_pos[rid] = [], [], []

        def visit(i):
            key, names, d = wins[i]
            rec = self._node(key, names, d, rid)
            self.read_nodes[rid].append(rec.hash)
            self.read_dirs[rid].append(d)
            self.read_pos[rid].append(wpos[i])
            rec.cov += 1
            return rec

        for g in range(n_win - 1):
            s = visit(g)
            key_t, names_t, d_t = wins[g + 1]
            t = self._node(key_t, names_t, d_t, rid)
            d_s = wins[g][2]
            fwd = self._stored_edge(s, t, d_s, d_t)
            rev = self._stored_edge(t, s, -d_t, -d_s)
            self._attach(s, fwd)
            self._attach(t, rev)
            fwd.cov += 1
            rev.cov += 1
        visit(n_win - 1)

    def _neighbours(self, node):
        return [self.edges[h].tgt for h in node.fw + node.bw]

    def _label_components(self):
        seen = set()
        comp = 0
        for nh, start in self.nodes.items():
            if nh in seen:
                continue
            comp += 1
            stack = [start]
            seen.add(nh)
            while stack:
                n = stack.pop()
                n.comp = comp
                for m in self._neighbours(n):
                    if m.hash not in seen:
                        seen.add(m.hash)
                        stack.append(m)

    # ---- removal ----------------------------------------------------------------
    def _remove_edge(self, eh):
        e = self.edges.get(eh)
        if e is None:
            return
        (e.src.fw if e.sd == 1 else e.src.bw).remove(eh)
        del self.edges[eh]

    def _remove_node(self, node):
        assert node.hash in self.nodes, "This node is not in the graph"
        for rid in node.reads:
            keep = [h != node.hash for h in self.read_nodes[rid]]
            for lst in (self.read_nodes, self.read_dirs, self.read_pos):
                lst[rid] = [v if kp else None for v, kp in zip(lst[rid], keep)]
            self.to_correct.add(rid)
        for eh in set(node.fw + node.bw):
            tgt = self.edges[eh].tgt
            out = [h for h in node.fw + node.bw if self.edges[h].tgt is tgt]
            back = [h for h in tgt.fw + tgt.bw if self.edges[h].tgt is node]
            assert out and back
            if len(out) > 1 or len(back) > 1:
                # the reference hands lists to remove_edge here and dies on `list in dict`
                raise TypeError("unhashable type: 'list'")
            self._remove_edge(out[0])
            self._remove_edge(back[0])
        del self.nodes[node.hash]

    def filter_graph(self, min_node_cov, min_edge_cov):
        self.min_node_cov, self.min_edge_cov = min_node_cov, min_edge_cov
        doomed = [n for n in self.nodes.values() if not n.cov > min_node_cov - 1]
        doomed_ids = {id(n) for n in doomed}
        doomed_edges = [
            e.hash for e in self.edges.values()
            if (not e.cov > min_edge_cov - 1) or id(e.src) in doomed_ids or id(e.tgt) in doomed_ids
        ]
        for eh in doomed_edges:
            self._remove_edge(eh)
        for n in doomed:
            self._remove_node(n)
        return self

    def remove_low_coverage_components(self, min_component_cov):
        comps = sorted({n.comp for n in self.nodes.values()})
        for c in comps:
            members = [n for n in self.nodes.values() if n.comp == c]
            if all(n.cov < min_component_cov for n in members):
                for n in members:
                    self._remove_node(n)

    def remove_nodes(self, indices):
        """remove_node, one at a time, for the nodes at these positions of the current node order (upstream's loop
        in remove_short_linear_paths / remove_non_AMR_associated_nodes).  Upstream raises TypeError half way through
        and leaves the graph partly edited; here the graph is restored, as the library leaves it unchanged."""
        nodes = list(self.nodes.values())
        doomed = [nodes[i] for i in sorted(set(int(i) for i in indices))]
        saved = copy.deepcopy(self.__dict__)
        try:
            for n in doomed:
                self._remove_node(n)
        except TypeError:
            self.__dict__ = saved
            raise

    # ---- array view -------------------------------------------------------------
    def vocabulary(self):
        """gene names ordered by ascending SHA-256 int; rank = index + 1"""
        names = {}
        for rid in self.read_ids:
            for c in self.reads_in[rid]:
                n, _ = parse_call(c)
                if n not in names:
                    names[n] = self._gene_hash.get(n) or sha_int(n)
        return sorted(names, key=names.get)

    def arrays(self, vocabulary=None):
        vocab = self.vocabulary() if vocabulary is None else vocabulary
        rank = {n: i + 1 for i, n in enumerate(vocab)}
        k = self.k
        nodes = list(self.nodes.values())
        nidx = {n.hash: i for i, n in enumerate(nodes)}
        edges = list(self.edges.values())
        eidx = {e.hash: i for i, e in enumerate(edges)}
        ridx = {r: i for i, r in enumerate(self.read_ids)}
        R = len(self.read_ids)

        def csr(lists, conv):
            off = np.zeros(len(lists) + 1, np.int64)
            flat = []
            for i, l in enumerate(lists):
                flat.extend(conv(x) for x in l)
                off[i + 1] = len(flat)
            return off, np.asarray(flat, np.int32).reshape(-1)

        out = {}
        out["k"] = np.int32(k)
        out["node_key"] = np.asarray(
            [[rank[nm] * st for nm, st in n.names] for n in nodes], np.int32).reshape(len(nodes), max(k, 0))
        out["node_cov"] = np.asarray([n.cov for n in nodes], np.uint32)
        out["node_dir"] = np.asarray([n.first_dir for n in nodes], np.int8)
        out["node_comp"] = np.asarray([n.comp for n in nodes], np.uint32)
        out["node_reads_off"], out["node_reads"] = csr([n.reads for n in nodes], ridx.__getitem__)
        out["fw_off"], out["fw_edges"] = csr([n.fw for n in nodes], eidx.__getitem__)
        out["bw_off"], out["bw_edges"] = csr([n.bw for n in nodes], eidx.__getitem__)
        out["edge_src"] = np.asarray([nidx[e.src.hash] for e in edges], np.int32)
        out["edge_tgt"] = np.asarray([nidx[e.tgt.hash] for e in edges], np.int32)
        out["edge_sd"] = np.asarray([e.sd for e in edges], np.int8)
        out["edge_td"] = np.asarray([e.td for e in edges], np.int8)
        out["edge_cov"] = np.asarray([e.cov for e in edges], np.uint32)
        win_off = np.zeros(R + 1, np.int64)
        wn, wd, ws, we = [], [], [], []
        for i, rid in enumerate(self.read_ids):
            hs = self.read_nodes.get(rid, [])
            for h, d, p in zip(hs, self.read_dirs.get(rid, []), self.read_pos.get(rid, [])):
                wn.append(-1 if h is None else nidx[h])
                wd.append(0 if d is None else d)
                ws.append(-1 if p is None else p[0])
                we.append(-1 if p is None else p[1])
            win_off[i + 1] = len(wn)
        out["win_off"] = win_off
        out["win_node"] = np.asarray(wn, np.int32).reshape(-1)
        out["win_dir"] = np.asarray(wd, np.int8).reshape(-1)
        out["win_start"] = np.asarray(ws, np.int32).reshape(-1)
        out["win_end"] = np.asarray(we, np.int32).reshape(-1)
        out["is_short"] = np.asarray([r in self.short_reads for r in self.read_ids], np.uint8)
        out["to_correct"] = np.asarray([r in self.to_correct for r in self.read_ids], np.uint8)
        return out


# ---- array-level helpers shared by tests / golden generation --------------------------------
ARRAY_FIELDS = (
    "node_key", "node_cov", "node_dir", "node_comp", "node_reads_off", "node_reads",
    "fw_off", "fw_edges", "bw_off", "bw_edges",
    "edge_src", "edge_tgt", "edge_sd", "edge_td", "edge_cov",
    "win_off", "win_node", "win_dir", "win_start", "win_end", "is_short", "to_correct",
)

_DTYPES = {
    "node_key": np.int32, "node_cov": np.uint32, "node_dir": np.int8, "node_comp": np.uint32,
    "node_reads_off": np.int64, "node_reads": np.int32, "fw_off": np.int64, "fw_edges": np.int32,
    "bw_off": np.int64, "bw_edges": np.int32, "edge_src": np.int32, "edge_tgt": np.int32,
    "edge_sd": np.int8, "edge_td": np.int8, "edge_cov": np.uint32, "win_off": np.int64,
    "win_node": np.int32, "win_dir": np.int8, "win_start": np.int32, "win_end": np.int32,
    "is_short": np.uint8, "to_correct": np.uint8,
}


def digest_arrays(arrs, fields=ARRAY_FIELDS) -> dict:
    """SHA-256 of each field's little-endian bytes (dtype-normalised) + a digest of digests."""
    out = {}
    for f in fields:
        a = np.ascontiguousarray(np.asarray(arrs[f]).astype(_DTYPES[f], copy=False))
        out[f] = hashlib.sha256(a.tobytes()).hexdigest()
    out["all"] = hashlib.sha256("".join(out[f] for f in fields).encode()).hexdigest()
    return out


def summary(arrs) -> dict:
    return {
        "nodes": int(len(arrs["node_cov"])), "edges": int(len(arrs["edge_cov"])),
        "windows": int(len(arrs["win_node"])), "sum_node_cov": int(arrs["node_cov"].sum()),
        "sum_edge_cov": int(arrs["edge_cov"].sum()), "short_reads": int(arrs["is_short"].sum()),
        "components": int(len(set(arrs["node_comp"].tolist()))),
        "incidences": int(len(arrs["node_reads"])), "none_windows": int((arrs["win_node"] < 0).sum()),
        "reads_to_correct": int(arrs["to_correct"].sum()),
    }


def diff_arrays(a, b, fields=ARRAY_FIELDS):
    """names of fields that differ (shape or content)"""
    bad = []
    for f in fields:
        x, y = np.asarray(a[f]), np.asarray(b[f])
        if x.shape != y.shape or not np.array_equal(x.astype(np.int64), y.astype(np.int64)):
            bad.append(f)
    return bad


def build_vocabulary(reads) -> list:
    """unique gene names of a {read_id: ['+g', ...]} dict, ascending SHA-256 int (rank = index + 1)"""
    hashes = {}
    for calls in reads.values():
        for c in calls:
            n, _ = parse_call(c)
            if n not in hashes:
                hashes[n] = sha_int(n)
    return sorted(hashes, key=hashes.get)


def encode_reads(reads, vocabulary, positions=None):
    """dict of string calls -> (signed int32 ids, int64 CSR offsets, pos_start, pos_end)"""
    rank = {n: i + 1 for i, n in enumerate(vocabulary)}
    ids, off, ps, pe = [], [0], [], []
    for rid, calls in reads.items():
        for c in calls:
            n, s = parse_call(c)
            ids.append(rank[n] * s)
        if positions:
            for a, b in positions[rid]:
                ps.append(a)
                pe.append(b)
        off.append(len(ids))
    ids = np.asarray(ids, np.int32).reshape(-1)
    off = np.asarray(off, np.int64)
    if positions:
        return ids, off, np.asarray(ps, np.int32).reshape(-1), np.asarray(pe, np.int32).reshape(-1)
    return ids, off, None, None
