"""GeneMerGraph: drop-in for upstream ``amira.construct_graph.GeneMerGraph`` on the graph-build path.

The constructor (upstream construct_graph.py:31-102), ``filter_graph`` (:523-540) and
``remove_low_coverage_components`` (:950-958) run on the GPU through the C ABI in
``include/amira_gmg.h``; this module encodes the read dict, calls the library and materialises the
exported arrays into the dictionaries and ``Node`` / ``Edge`` objects downstream code reaches into:
``_nodes`` / ``_edges`` keyed by upstream's SHA-256 integers in upstream's insertion order,
``_readNodes`` / ``_readNodeDirections`` / ``_readNodePositions`` per read, ``_shortReads``,
``_readsToCorrect``.  The single-object accessors and mutators of the same surface
(``add_node``, ``remove_node``, ...) are plain host code over those objects, as upstream's are.

The host objects are materialised LAZILY: the constructor only encodes the reads and enqueues the device
build; the dictionaries and ``Node`` / ``Edge`` objects are created the first time something reaches for
``_nodes`` / ``_edges`` / the per-read lists.  Filters, component removal, the coverage statistics, the junk-read
and valid-read selections and the GML writer work on the device arrays and never need them.

There is no CPU build: without ``libamira_gmg.so`` or without a CUDA device construction fails.

To run upstream's own correction / path-finding methods on top of the GPU build, see
``bind_upstream`` below and INTEGRATION.md.
"""
from __future__ import annotations

import os
import statistics
import weakref
import zlib

import numpy as np

from . import _keys, _lib, encode
from .construct_edge import Edge, edge_key
from .construct_gene import Gene, convert_int_strand_to_string, hashlib_hash
from .construct_gene_mer import GeneMer
from .construct_node import Node
from .device_graph import DeviceGraph

_HANDLES: dict = {}      # device index -> DeviceGraph shared by the graphs built on that device


def _device_index(device) -> int:
    if device is None:
        return int(os.environ.get("AMIRA_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    return int(device)


def _handle(device: int) -> DeviceGraph:
    h = _HANDLES.get(device)
    if h is None:
        h = _HANDLES[device] = DeviceGraph(device)
        h.owner = None
    return h


def _host(x) -> np.ndarray:
    """a numpy array, or a device tensor copied to one"""
    return x if isinstance(x, np.ndarray) else x.cpu().numpy()


def _union(a, b):
    """a | b for per-read flags, on b's device when b is a device tensor"""
    if isinstance(a, np.ndarray) and not isinstance(b, np.ndarray):
        import torch
        a = torch.from_numpy(a).to(b.device)
    return a | b


class _Classes:
    """the element classes a graph is materialised with (ours, or upstream's when bound)"""
    Gene, GeneMer, Node, Edge = Gene, GeneMer, Node, Edge

    @staticmethod
    def make_gene(name, strand):
        return Gene.from_parts(name, strand)

    @staticmethod
    def make_genemer(canonical, rc, direction, node_hash):
        return GeneMer.from_canonical(canonical, rc, direction, node_hash)

    @staticmethod
    def make_node(genemer, node_hash, cov, reads, comp):
        return Node.from_arrays(genemer, node_hash, cov, reads, comp)

    @staticmethod
    def make_edge(src, tgt, sd, td, cov):
        e = Edge(src, tgt, sd, td)
        e.edgeCoverage = cov
        return e


_LAZY_ATTRS = ("_nodes", "_edges", "_readNodes", "_readNodeDirections", "_readNodePositions", "_shortReads",
               "_readsToCorrect")


def _lazy_property(name):
    slot = "_m" + name

    def get(self):
        if self.__dict__.get("_lazy"):
            self._materialise_now()
        return self.__dict__[slot]

    def set_(self, value):
        self.__dict__[slot] = value

    return property(get, set_)


class GeneMerGraph:
    _cls = _Classes
    for _a in _LAZY_ATTRS:
        locals()[_a] = _lazy_property(_a)
    del _a

    def __init__(self, readDict, kmerSize, gene_positions=None, device=None):
        # an encode.EncodedReads in place of the dict: the strings were parsed once, reuse the CSR
        self._lazy = False
        self._encoded = readDict if isinstance(readDict, encode.EncodedReads) else None
        if self._encoded is not None:
            if gene_positions is not None and gene_positions is not self._encoded.positions:
                # explicit positions win: encode them against the same reads (the cached CSR has none / others)
                self._encoded = encode.EncodedReads(self._encoded.reads, gene_positions)
            gene_positions = self._encoded.positions
            readDict = self._encoded.reads
        self._reads = readDict
        self._kmerSize = kmerSize
        self._minNodeCoverage = 1
        self._minEdgeCoverage = 1
        self._genePositions = gene_positions
        self._nodes = {}
        self._edges = {}
        self._readNodes = {}
        self._readNodeDirections = {}
        self._readNodePositions = {}
        self._shortReads = {}
        self._readsToCorrect = set()
        self._device = _device_index(device)
        self._device_synced = False      # device state == host objects
        self._node_order = []            # node hashes in device index order
        self._edge_order = []
        self._node_objs = []             # Node objects in device index order
        self._read_ids = []
        self._win_off = None
        self._device_ops = ()
        self._index_cache = None         # node hash -> device index of a materialised device graph
        self.timings = {}
        _lib.load()                      # fail loudly if the CUDA library is missing
        if len(readDict) > 0:
            self._build_on_device()

    # ------------------------------------------------------------------ device build
    def _encode(self):
        if self._encoded is not None:
            e = self._encoded
            return e.vocab, e.ids, e.off, e.pos_start, e.pos_end
        reads = self._reads
        vocab = encode.Vocabulary(encode.collect_names(reads))
        positions = self._genePositions if self._genePositions else None
        ids, off, ps, pe = encode.encode_reads(reads, vocab, positions)
        return vocab, ids, off, ps, pe

    def _build_on_device(self):
        vocab, ids, off, ps, pe = self._encode()
        h = _handle(self._device)
        h.owner = None
        if self._encoded is not None and hasattr(h, "build_resident"):
            h.build_resident(self._encoded, int(self._kmerSize), self._device)
        else:
            h.build(ids, off, int(self._kmerSize), ps, pe)
        self._adopt_build(h, vocab, ids, off)

    def _adopt_build(self, h, vocab, ids, off):
        """make the build the handle holds, of this graph's reads (vocab, host ids / off), this graph's lazy device copy"""
        self._vocab = vocab
        self._csr_fingerprint = (len(ids), int(off[-1]) if len(off) else 0, zlib.crc32(np.ascontiguousarray(ids).tobytes()))
        self._read_len = np.diff(off)
        h.owner = weakref.ref(self)
        self._read_ids = list(self._reads)
        self._device_synced = True
        self._lazy = True                # host objects on first use (_materialise_now)

    def _materialise_now(self):
        """create the host dictionaries and objects from the device arrays (first access to _nodes / _edges / ...)"""
        if not self.__dict__.get("_lazy"):
            return
        self._lazy = False
        h = self._require_device_state()
        # 10^5..10^6 long-lived objects are created in one go: the cyclic collector would re-scan them generation by
        # generation on the way (measured on C2: 1.3 s -> 0.8 s without it); nothing here can form garbage cycles
        import gc
        was_enabled = gc.isenabled()
        gc.disable()
        try:
            self._materialise(h.arrays(), self._vocab)
        finally:
            if was_enabled:
                gc.enable()

    def _arrays(self, *fields):
        """current device arrays of this graph (no host objects involved)"""
        h = self._require_device_state()
        a = h.arrays()
        return a if not fields else tuple(a[f] for f in fields)

    def _materialise(self, a, vocab):
        C = self._cls
        reads = self._reads
        k = int(self._kmerSize)
        read_ids = list(reads)
        self._read_ids = read_ids
        V = len(vocab)
        # one Gene object per signed id, and its signed SHA integer
        genes = np.empty(2 * V + 1, object)
        for r, name in enumerate(vocab.names, 1):
            genes[V + r] = C.make_gene(name, 1)
            genes[V - r] = C.make_gene(name, -1)
        key = a["node_key"].astype(np.int64)
        n_nodes = key.shape[0]
        canon_rows = genes[key + V].tolist() if n_nodes else []
        rc_rows = genes[V - key[:, ::-1]].tolist() if n_nodes else []
        node_hashes, node_sha = _keys.node_keys(key, vocab)
        rid_arr = np.empty(len(read_ids), object)
        rid_arr[:] = read_ids
        nr_off = a["node_reads_off"].tolist()
        nr = rid_arr[a["node_reads"]].tolist() if len(a["node_reads"]) else []
        cov = a["node_cov"].tolist()
        ndir = a["node_dir"].tolist()
        comp = a["node_comp"].tolist()
        nodes = self._nodes
        node_objs = []
        for i in range(n_nodes):
            nh = node_hashes[i]
            gm = C.make_genemer(canon_rows[i], rc_rows[i], ndir[i], nh)
            node = C.make_node(gm, nh, cov[i], nr[nr_off[i]:nr_off[i + 1]], comp[i])
            nodes[nh] = node
            node_objs.append(node)
        self._node_order = node_hashes
        self._node_objs = node_objs
        # edges
        src, tgt = a["edge_src"].tolist(), a["edge_tgt"].tolist()
        sd, td, ecov = a["edge_sd"].tolist(), a["edge_td"].tolist(), a["edge_cov"].tolist()
        edges = self._edges
        edge_hashes = _keys.edge_keys(node_hashes, node_sha, a["edge_src"], a["edge_tgt"], a["edge_sd"], a["edge_td"])
        for j, eh in enumerate(edge_hashes):
            edges[eh] = C.make_edge(node_objs[src[j]], node_objs[tgt[j]], sd[j], td[j], ecov[j])
        self._edge_order = edge_hashes
        if edge_hashes:
            eh_arr = np.empty(len(edge_hashes), object)
            eh_arr[:] = edge_hashes
            fw = eh_arr[a["fw_edges"]].tolist()
            bw = eh_arr[a["bw_edges"]].tolist()
            fo, bo = a["fw_off"].tolist(), a["bw_off"].tolist()
            for i, node in enumerate(node_objs):
                node.forwardEdgeHashes = fw[fo[i]:fo[i + 1]]
                node.backwardEdgeHashes = bw[bo[i]:bo[i + 1]]
        # per-read lists (windows of removed nodes are None: the arrays may come from a filtered device graph)
        woff = a["win_off"].tolist()
        self._win_off = woff
        win = a["win_node"]
        gone = win < 0
        any_gone = bool(gone.any())
        if n_nodes:
            nh_arr = np.empty(n_nodes + 1, object)
            nh_arr[:n_nodes] = node_hashes
            nh_arr[n_nodes] = None
            wn = nh_arr[np.where(gone, n_nodes, win)].tolist()
        else:
            wn = [None] * len(win)
        wd = a["win_dir"].tolist()
        if any_gone:
            wd = [None if g else d for d, g in zip(wd, gone.tolist())]
        has_pos = bool(self._genePositions)
        if has_pos:
            wp = list(zip(a["win_start"].tolist(), a["win_end"].tolist()))
            if any_gone:
                wp = [None if g else p for p, g in zip(wp, gone.tolist())]
        short = a["is_short"].tolist()
        rn, rd, rp = self._readNodes, self._readNodeDirections, self._readNodePositions
        for i, rid in enumerate(read_ids):
            if short[i]:
                self._shortReads[rid] = reads[rid]
                continue
            lo, hi = woff[i], woff[i + 1]
            rn[rid] = wn[lo:hi]
            rd[rid] = wd[lo:hi]
            if has_pos and self._genePositions[rid]:
                rp[rid] = wp[lo:hi]
            else:
                rp[rid] = [None] * (hi - lo)
        self._readsToCorrect.update(rid for rid, c in zip(read_ids, a["to_correct"].tolist()) if c)

    def _require_device_state(self):
        """the device copy of this graph, rebuilt if another graph has used the handle since"""
        if not self._device_synced:
            raise RuntimeError(
                "this graph was modified on the host after its device build; the GPU filter works on the "
                "device copy (there is no CPU filter path). Rebuild it with GeneMerGraph(reads, k) first.")
        h = _handle(self._device)
        if h.owner is None or h.owner() is not self:
            vocab, ids, off, ps, pe = self._encode()
            fp = (len(ids), int(off[-1]) if len(off) else 0, zlib.crc32(np.ascontiguousarray(ids).tobytes()))
            if vocab.names != self._vocab.names or fp != self._csr_fingerprint:
                raise RuntimeError("the read dict of this graph changed since it was built; rebuild it first")
            h.owner = None
            h.build(ids, off, int(self._kmerSize), ps, pe)
            for op, args in self._device_ops:
                getattr(h, op)(*args)
            h.owner = weakref.ref(self)
        return h

    def _apply_device_removal(self, h):
        """mirror the device's last removal on the host objects (same deletions upstream performs)"""
        self._index_cache = None
        if self.__dict__.get("_lazy"):
            return                       # nothing materialised yet: the arrays are the graph
        node_keep, edge_keep = h.filter_masks()
        if node_keep.all() and edge_keep.all():
            return
        edges, nodes = self._edges, self._nodes
        for j in np.flatnonzero(~edge_keep).tolist():
            eh = self._edge_order[j]
            e = edges.pop(eh)
            src = e.get_sourceNode()
            lst = src.forwardEdgeHashes if e.get_sourceNodeDirection() == 1 else src.backwardEdgeHashes
            lst.remove(eh)
        self._edge_order = [eh for eh, kp in zip(self._edge_order, edge_keep.tolist()) if kp]
        gone = np.flatnonzero(~node_keep).tolist()
        if not gone:
            return
        affected = set()
        for i in gone:
            node = nodes.pop(self._node_order[i])
            affected.update(node.get_list_of_reads())
        self._node_order = [nh for nh, kp in zip(self._node_order, node_keep.tolist()) if kp]
        self._node_objs = [n for n, kp in zip(self._node_objs, node_keep.tolist()) if kp]
        # per-read lists: windows of removed nodes become None (remove_node_from_reads, :442-461)
        a = h.arrays_reads_only()
        wn = a["win_node"]
        woff = self._win_off
        rn, rd, rp = self._readNodes, self._readNodeDirections, self._readNodePositions
        ridx = {r: i for i, r in enumerate(self._read_ids)}
        for rid in affected:
            i = ridx[rid]
            mask = (wn[woff[i]:woff[i + 1]] < 0).tolist()
            rn[rid] = [None if m else v for v, m in zip(rn[rid], mask)]
            rd[rid] = [None if m else v for v, m in zip(rd[rid], mask)]
            rp[rid] = [None if m else v for v, m in zip(rp[rid], mask)]
        self._readsToCorrect.update(affected)

    # ------------------------------------------------------------------ GPU-backed operations
    def filter_graph(self, minNodeCoverage: int, minEdgeCoverage: int):
        """upstream construct_graph.py:523-540"""
        minNodeCoverage = self.set_minNodeCoverage(minNodeCoverage)
        minEdgeCoverage = self.set_minEdgeCoverage(minEdgeCoverage)
        if self.get_total_number_of_nodes() == 0:
            return self
        h = self._require_device_state()
        h.filter_graph(max(int(minNodeCoverage), 0), max(int(minEdgeCoverage), 0))
        self._device_ops = self._device_ops + (("filter_graph", (max(int(minNodeCoverage), 0), max(int(minEdgeCoverage), 0))),)
        self._apply_device_removal(h)
        return self

    def remove_low_coverage_components(self, min_component_coverage):
        """upstream construct_graph.py:950-958"""
        if self.get_total_number_of_nodes() == 0:
            return
        h = self._require_device_state()
        h.remove_low_coverage_components(max(int(min_component_coverage), 0))
        self._device_ops = self._device_ops + (("remove_low_coverage_components", (max(int(min_component_coverage), 0),)),)
        self._apply_device_removal(h)

    # ------------------------------------------------------------------ accessors
    def get_reads(self):
        return self._reads

    def get_short_read_annotations(self):
        return self._shortReads

    def get_gene_positions(self):
        return self._genePositions

    def get_short_read_gene_positions(self):
        return {r: self._genePositions[r] for r in self._shortReads}

    def get_readNodes(self):
        return self._readNodes

    def get_readNodeDirections(self):
        return self._readNodeDirections

    def get_readNodePositions(self):
        return self._readNodePositions

    def get_kmerSize(self) -> int:
        return self._kmerSize

    def get_minEdgeCoverage(self) -> int:
        return self._minEdgeCoverage

    def get_minNodeCoverage(self) -> int:
        return self._minNodeCoverage

    def get_nodes(self):
        return self._nodes

    def get_edges(self):
        return self._edges

    def get_reads_to_correct(self) -> set:
        return self._readsToCorrect

    def all_nodes(self):
        yield from self._nodes.values()

    def get_reads_for_nodes(self, list_of_nodes) -> set:
        reads = set()
        for node_hash in list_of_nodes:
            reads.update(self._nodes[node_hash].get_list_of_reads())
        return reads

    def get_nodes_containing_read(self, readId: str):
        return [self._nodes[h] for h in self._readNodes[readId] if h in self._nodes]

    def get_node_by_hash(self, nodeHash: int):
        return self._nodes[nodeHash]

    def get_edge_by_hash(self, edgeHash: int):
        return self._edges[edgeHash]

    def get_node(self, geneMer):
        nodeHash = geneMer.__hash__()
        assert nodeHash in self._nodes, "This gene-mer is not in the graph"
        return self._nodes[nodeHash]

    def get_nodes_containing(self, geneOfInterest: str):
        assert not (geneOfInterest[0] == "+" or geneOfInterest[0] == "-"), \
            "Strand information cannot be present for any specified genes"
        assert isinstance(geneOfInterest, str), "Gene of interest is the wrong type"
        if self._on_device():
            nodes = self._nodes                                   # materialises; keeps _node_objs in device order
            rank = self._gene_ranks([geneOfInterest])
            if not rank:
                return []
            flags = self._require_device_state().nodes_containing(rank)
            return [self._node_objs[i] for i in np.flatnonzero(flags).tolist()]
        return [n for n in self._nodes.values()
                if geneOfInterest in [g.get_name() for g in n.get_canonical_geneMer()]]

    def _gene_ranks(self, names) -> list:
        """SHA ranks (1..V) of the gene names that occur in this graph's vocabulary"""
        if getattr(self, "_rank_of", None) is None:
            self._rank_of = {n: i + 1 for i, n in enumerate(self._vocab.names)}
        return [self._rank_of[n] for n in names if n in self._rank_of]

    def get_AMR_nodes(self, listOfGenes):
        """upstream construct_graph.py:963-972: {node hash: node} of the nodes that contain any of the genes"""
        if self._on_device():
            nodes = self._nodes
            h = self._require_device_state()
            out = {}
            for g in listOfGenes:                  # upstream's dict order: by gene, then by node
                for r in self._gene_ranks([g]):
                    for i in np.flatnonzero(h.nodes_containing([r])).tolist():
                        out[self._node_order[i]] = self._node_objs[i]
            return out
        out = {}
        for g in listOfGenes:
            for node in self.get_nodes_containing(g):
                out[node.__hash__()] = node
        return out

    def remove_non_AMR_associated_nodes(self, genesOfInterest):
        """upstream construct_graph.py:2941-2959: drop every node that shares no read with a node holding one of the
        genes.  On the device: flag nodes, mark their reads, keep the nodes that touch a marked read, compact."""
        if self._on_device():
            for g in genesOfInterest:
                assert not (g[0] == "+" or g[0] == "-"), "Strand information cannot be present for any specified genes"
            h = self._require_device_state()
            ranks = self._gene_ranks(list(genesOfInterest))
            h.remove_nodes_without_reads_of(ranks)
            self._device_ops = self._device_ops + (("remove_nodes_without_reads_of", (tuple(ranks),)),)
            self._apply_device_removal(h)
            return
        readsOfInterest = set()
        for g in genesOfInterest:
            for node in self.get_nodes_containing(g):
                readsOfInterest.update(node.get_reads())
        doomed = [n for n in self._nodes.values() if not readsOfInterest.intersection(n.get_list_of_reads())]
        for node in doomed:
            self.remove_node(node)

    # ------------------------------------------------------------------ linear paths (upstream :722-861, 679-720)
    def _linear_steps(self) -> dict:
        """per node and side of a graph edited on the host: upstream's one step of a linear-path walk (next node index,
        entry direction, extend flag) and the node degrees, from the host objects (device graphs walk on the device:
        amira_gmg_linear_walks)"""
        nodes = self._nodes
        order = list(nodes)
        index = {h: i for i, h in enumerate(order)}
        st = {"index": index, "hash": order, "degree": [self.get_degree(n) for n in nodes.values()]}
        for side, getter in (("fw", "get_forward_edge_hashes"), ("bw", "get_backward_edge_hashes")):
            nxt, dr, ext = [], [], []
            for h, node in nodes.items():
                eh = getattr(node, getter)()
                take = len(eh) == 1 if side == "fw" else len(eh) > 0
                if not take:
                    nxt.append(-1); dr.append(0); ext.append(0)
                    continue
                e = self._edges[eh[0]]
                t = e.get_targetNode()
                nxt.append(index[t.__hash__()])
                dr.append(e.get_targetNodeDirection())
                ext.append(int(self.get_degree(t) in (1, 2) and t != node))
            st[side + "_next"], st[side + "_dir"], st[side + "_ext"] = nxt, dr, ext
        return st

    def _walk(self, st, start: int, first_side: str, backward: bool, want_branched: bool) -> list:
        """get_forward_path_from_node / get_backward_path_from_node on node indices"""
        path = [start]
        ext, nx, d = st[first_side + "_ext"][start], st[first_side + "_next"][start], st[first_side + "_dir"][start]
        while ext:
            if path[-1 if backward else 0] == nx:
                break                                   # (upstream compares with the far end of the list and stops)
            if backward:
                path.insert(0, nx)
            else:
                path.append(nx)
            side = ("bw" if d == -1 else "fw") if backward else ("fw" if d == 1 else "bw")
            ext, nx, d = st[side + "_ext"][nx], st[side + "_next"][nx], st[side + "_dir"][nx]
        if want_branched and nx is not None and nx >= 0:
            if backward:
                path.insert(0, nx)
            else:
                path.append(nx)
        return path

    def _walks_over(self, st, states, want_branched: bool) -> tuple:
        """_walk from every state 2 * node + side (0 = forward list, 1 = backward list) of the step table `st`, without
        the start node -> (offsets, nodes), as amira_gmg_linear_walks returns them"""
        off, out = [0], []
        for s in np.asarray(states, np.int64).tolist():
            out.extend(self._walk(st, s >> 1, "bw" if s & 1 else "fw", False, want_branched)[1:])
            off.append(len(out))
        return np.asarray(off, np.int64), np.asarray(out, np.int64)

    def _device_walks(self, h, states, want_branched: bool) -> tuple:
        """linear walks on the device graph (amira_gmg_linear_walks).  A handle without them -- the oracle-backed test
        double the CPU tests build with -- is walked with _walk over its step table."""
        if hasattr(h, "linear_walks"):
            return h.linear_walks(states, want_branched)
        return self._walks_over({f: v.tolist() for f, v in h.linear_steps().items()}, states, want_branched)

    def _device_walk(self, node, side: int, want_branched: bool) -> list:
        """node hashes of the device walk from one side (0 = forward list, 1 = backward list) of a node, the node first"""
        self._nodes                                     # the arguments are node objects: materialised, in device order
        if self._index_cache is None:
            self._index_cache = {h: i for i, h in enumerate(self._node_order)}
        i = self._index_cache[node.__hash__()]
        _, walk = self._device_walks(self._require_device_state(), [2 * i + side], want_branched)
        order = self._node_order
        return [order[i]] + [order[j] for j in walk.tolist()]

    def get_forward_path_from_node(self, node, startDirection, wantBranchedNode=False) -> list:
        side = 0 if startDirection == 1 else 1
        if self._on_device():
            return self._device_walk(node, side, wantBranchedNode)
        st = self._linear_steps()
        i = st["index"][node.__hash__()]
        return [st["hash"][j] for j in self._walk(st, i, ("fw", "bw")[side], False, wantBranchedNode)]

    def get_backward_path_from_node(self, node, startDirection, wantBranchedNode=False) -> list:
        side = 1 if startDirection == -1 else 0
        if self._on_device():
            return self._device_walk(node, side, wantBranchedNode)[::-1]
        st = self._linear_steps()
        i = st["index"][node.__hash__()]
        return [st["hash"][j] for j in self._walk(st, i, ("fw", "bw")[side], True, wantBranchedNode)]

    def get_linear_path_for_node(self, node, wantBranchedNode=False) -> list:
        """upstream construct_graph.py:849-861"""
        d = node.get_geneMer().get_geneMerDirection()
        back = self.get_backward_path_from_node(node, -1 * d, wantBranchedNode)
        assert back[-1] == node.__hash__()
        fwd = self.get_forward_path_from_node(node, d, wantBranchedNode)
        assert fwd[0] == node.__hash__()
        return back[:-1] + [node.__hash__()] + fwd[1:]

    def remove_short_linear_paths(self, min_length, sample_genesOfInterest={}):
        """upstream construct_graph.py:679-720: dead ends (degree-1 nodes) whose linear path is shorter than min_length
        are removed unless the whole path is well covered, holds an AMR gene or is its whole component.  A device graph
        is walked on the device (amira_gmg_linear_walks) and trimmed in one device pass (amira_gmg_remove_nodes)
        without creating host objects; a graph edited on the host is walked over its objects."""
        if self._on_device():
            if self.get_total_number_of_nodes() == 0:
                return []
            h = self._require_device_state()
            degree = h.linear_steps()["degree"]
            cov, comp, ndir, key = self._arrays("node_cov", "node_comp", "node_dir", "node_key")
            ranks = self._gene_ranks(list(sample_genesOfInterest))
            amr = h.nodes_containing(ranks) if ranks else np.zeros(len(cov), bool)
            removed = self._short_path_nodes(min_length, degree, cov, comp.astype(np.int64), ndir, amr,
                                             lambda states: self._device_walks(h, states, False))
            if not len(removed):
                return []
            hashes = _keys.node_keys(key[removed].astype(np.int64), self._vocab)[0]
            flags = np.zeros(len(cov), np.uint8)
            flags[removed] = 1
            h.remove_nodes(flags)
            self._device_ops = self._device_ops + (("remove_nodes", (flags,)),)
            self._apply_device_removal(h)
            return hashes
        st = self._linear_steps()
        nodes = self._nodes
        if not nodes:
            return []
        objs = list(nodes.values())
        codes = {}                                      # component ids (None: no component) -> 0, 1, ...
        comp = np.asarray([-1 if n.get_component() is None else codes.setdefault(n.get_component(), len(codes))
                           for n in objs], np.int64)
        AMR_nodes = self.get_AMR_nodes(sample_genesOfInterest)
        amr = np.asarray([nh in AMR_nodes for nh in st["hash"]], bool)
        removed = self._short_path_nodes(min_length, np.asarray(st["degree"]), np.asarray([n.get_node_coverage() for n in objs]),
                                         comp, np.asarray([n.get_geneMer().get_geneMerDirection() for n in objs]), amr,
                                         lambda states: self._walks_over(st, states, False))
        hashes = [st["hash"][i] for i in removed.tolist()]
        for nh in hashes:
            self.remove_node(nodes[nh])
        return hashes

    def _short_path_nodes(self, min_length, degree, cov, comp, ndir, amr, walks) -> np.ndarray:
        """the trimming policy of remove_short_linear_paths over node indices.  walks(states) -> (offsets, nodes) gives
        the linear walks from the states 2 * node + side; comp[i] = -1: node i has no component.  Returns the nodes to
        remove in upstream's order: component first seen, then path, then node along the path, each node once."""
        none = np.zeros(0, np.int64)
        tips = np.flatnonzero(degree == 1)
        if not len(tips):
            return none
        # get_linear_path_for_node: the backward walk (reversed), the node, the forward walk
        back = (ndir[tips] == 1).astype(np.int64)
        off, w = walks(np.stack([2 * tips + back, 2 * tips + 1 - back], 1).ravel())
        off, w = np.asarray(off, np.int64), np.asarray(w, np.int64)
        nb, nf = off[1::2] - off[0:-1:2], off[2::2] - off[1::2]
        q = np.flatnonzero(nb + 1 + nf < min_length)     # short paths, by tip
        if not len(q):
            return none
        plen = nb[q] + 1 + nf[q]
        start = np.concatenate([[0], np.cumsum(plen)[:-1]])
        pid = np.repeat(np.arange(len(q)), plen)          # path of every element, elements in path order
        p = np.arange(len(pid)) - start[pid]
        b = nb[q][pid]
        w_end = np.append(w, -1)
        bi = np.where(p < b, off[2 * q][pid] + b - 1 - p, len(w))
        fi = np.where(p > b, off[2 * q + 1][pid] + p - b - 1, len(w))
        node = np.where(p == b, tips[q][pid], np.where(p < b, w_end[bi], w_end[fi]))
        # paths whose every node is covered above 1.5 x the mean stay
        mean15 = self.get_mean_node_coverage() * 1.5
        kept = np.add.reduceat((cov[node] <= mean15).astype(np.int64), start) > 0
        # components in the order their first kept path was seen
        c = comp[tips[q]]
        kq = np.flatnonzero(kept)
        _, first, inv = np.unique(c[kq], return_index=True, return_inverse=True)
        rank = np.full(len(q), len(q), np.int64)
        rank[kq] = first[inv.ravel()]
        # a path that is its whole component stays
        n_nodes = len(degree)
        sizes = np.bincount(comp[comp >= 0], minlength=n_nodes)
        u = np.unique(pid * n_nodes + node)
        upid, unode = u // n_nodes, u % n_nodes
        in_comp = np.bincount(upid[comp[unode] == c[upid]], minlength=len(q))
        whole = (c >= 0) & (in_comp == sizes[np.maximum(c, 0)])
        go = kept & ~whole
        sel = np.flatnonzero(go[pid] & ~amr[node])
        seq = node[sel[np.argsort(rank[pid[sel]], kind="stable")]]
        _, first_at = np.unique(seq, return_index=True)
        return seq[np.sort(first_at)]

    # ------------------------------------------------------------------ compacted graph (no upstream counterpart)
    def compacted_unitigs(self) -> dict:
        """every maximal non-branching path as one unitig (include/amira_gmg.h, amira_gmg_unitigs), as numpy arrays:
        node_unitig / node_pos / node_orient per node in `_nodes` order; unitig_off / unitig_nodes (node indices in
        listed order), circular, cov_sum / cov_min / cov_max per unitig; edge_internal per edge in `_edges` order (1:
        the edge joins consecutive nodes of one unitig, 0: a junction).  A device graph is compacted on the device and
        stays lazy; a graph edited on the host is compacted from its objects."""
        if self._on_device():
            h = self._require_device_state()
            if hasattr(h, "unitigs"):
                return h.unitigs()
            return self._unitigs_over(h.arrays())
        return self._unitigs_over(self._unitig_index_arrays())

    def _unitig_index_arrays(self) -> dict:
        """the index arrays _unitigs_over and _links_over read, from the host objects: nodes in `_nodes` order, edges
        in `_edges` order, each node's forward / backward list as a CSR over edge indices"""
        nodes, edges = self._nodes, self._edges
        index = {nh: i for i, nh in enumerate(nodes)}
        eindex = {eh: j for j, eh in enumerate(edges)}
        es = list(edges.values())
        a = {"node_cov": np.asarray([n.get_node_coverage() for n in nodes.values()], np.int64),
             "edge_src": np.asarray([index[e.get_sourceNode().__hash__()] for e in es], np.int64),
             "edge_tgt": np.asarray([index[e.get_targetNode().__hash__()] for e in es], np.int64),
             "edge_sd": np.asarray([e.get_sourceNodeDirection() for e in es], np.int64),
             "edge_td": np.asarray([e.get_targetNodeDirection() for e in es], np.int64),
             "edge_cov": np.asarray([e.get_edge_coverage() for e in es], np.int64)}
        for side, getter in (("fw", "get_forward_edge_hashes"), ("bw", "get_backward_edge_hashes")):
            lists = [getattr(n, getter)() for n in nodes.values()]
            a[side + "_off"] = np.concatenate([[0], np.cumsum([len(x) for x in lists], dtype=np.int64)]).astype(np.int64)
            a[side + "_edges"] = np.asarray([eindex[eh] for x in lists for eh in x], np.int64)
        return a

    def _unitigs_over(self, a) -> dict:
        """amira_gmg_unitigs over index arrays (node_cov, edge_src / tgt / sd / td, fw_off / fw_edges, bw_off /
        bw_edges), by the same list ranking as csrc/unitigs.cuh: states s = 2 * node + side, succ(s), distances to
        the tail and running minima by pointer jumping, cycles cut at their smallest state"""
        N = len(a["node_cov"])
        S = 2 * N
        out = {"node_unitig": np.zeros(N, np.int32), "node_pos": np.zeros(N, np.int32), "node_orient": np.zeros(N, np.int8),
               "unitig_off": np.zeros(1, np.int64), "unitig_nodes": np.zeros(N, np.int32), "circular": np.zeros(0, np.uint8),
               "cov_sum": np.zeros(0, np.int64), "cov_min": np.zeros(0, np.uint32), "cov_max": np.zeros(0, np.uint32),
               "edge_internal": np.zeros(len(a["edge_src"]), np.uint8)}
        if N == 0:
            return out
        succ = self._unitig_succ(a)
        idx = np.arange(S, dtype=np.int64)
        rounds = int(S - 1).bit_length() + 1                                         # ceil(log2 S) + 1

        def rank(cut, mn=None):
            ptr, dist = np.where(cut, idx, succ), (~cut).astype(np.int64)
            for _ in range(rounds):
                if mn is not None:
                    mn = np.minimum(mn, mn[ptr])
                dist = np.minimum(dist + dist[ptr], S)
                ptr = ptr[ptr]
            return ptr, dist, mn

        ptr, dist, mn = rank(succ < 0, idx)
        cyc = succ[ptr] >= 0
        if cyc.any():
            dist = rank((succ < 0) | (cyc & (mn == idx)))[1]
        nodes = np.arange(N, dtype=np.int64)
        cm = np.minimum(mn[0::2], mn[1::2] ^ 1)          # the smallest state of the chain of 2n
        m, s = cm >> 1, 2 * nodes + (cm & 1)              # the unitig's smallest node, the state n is listed through
        heads = np.flatnonzero(m == nodes)
        uid = np.zeros(N, np.int64)
        uid[heads] = np.arange(len(heads))
        circ = cyc[2 * heads]
        length = np.where(circ, dist[np.maximum(succ[2 * heads], 0)] + 1, dist[2 * heads] + dist[2 * heads + 1] + 1)
        off = np.concatenate([[0], np.cumsum(length)]).astype(np.int64)
        unit, pos = uid[m], dist[s ^ 1]
        order = np.zeros(N, np.int64)
        order[off[unit] + pos] = nodes
        cov = np.asarray(a["node_cov"], np.int64)[order]
        src = np.asarray(a["edge_src"], np.int64)
        out.update(node_unitig=unit.astype(np.int32), node_pos=pos.astype(np.int32),
                   node_orient=np.where(s & 1, -1, 1).astype(np.int8), unitig_off=off, unitig_nodes=order.astype(np.int32),
                   circular=circ.astype(np.uint8), cov_sum=np.add.reduceat(cov, off[:-1]),
                   cov_min=np.minimum.reduceat(cov, off[:-1]).astype(np.uint32),
                   cov_max=np.maximum.reduceat(cov, off[:-1]).astype(np.uint32),
                   edge_internal=(succ[2 * src + (np.asarray(a["edge_sd"]) < 0)] >= 0).astype(np.uint8))
        return out

    @staticmethod
    def _unitig_succ(a) -> np.ndarray:
        """succ of every state s = 2 * node + side over index arrays (csrc/unitigs.cuh), -1 where there is none: list
        `side` of the node holds one edge (-> v, td), v is another node, and v's entering list holds one edge"""
        S = 2 * len(a["node_cov"])
        tgt, td = np.asarray(a["edge_tgt"], np.int64), np.asarray(a["edge_td"], np.int64)
        size, one = GeneMerGraph._list_sizes(a)
        st = np.flatnonzero(one >= 0)
        v, leave = tgt[one[st]], (td[one[st]] != 1).astype(np.int64)
        ok = (v != st >> 1) & (size[2 * v + (1 - leave)] == 1)
        succ = np.full(S, -1, np.int64)
        succ[st[ok]] = 2 * v[ok] + leave[ok]
        return succ

    @staticmethod
    def _list_sizes(a) -> tuple:
        """over index arrays: size[s], the number of edges in the list of state s, and one[s], the edge of a one-edge
        list (-1 for the others)"""
        size = np.stack([np.diff(a["fw_off"]), np.diff(a["bw_off"])], 1).ravel()
        one = np.full(len(size), -1, np.int64)
        for side, f in enumerate(("fw", "bw")):
            sel = np.flatnonzero(np.diff(a[f + "_off"]) == 1)
            one[2 * sel + side] = np.asarray(a[f + "_edges"], np.int64)[np.asarray(a[f + "_off"], np.int64)[sel]]
        return size, one

    def compacted_links(self) -> dict:
        """the junction edges of the compacted graph (include/amira_gmg.h, amira_gmg_unitig_links), one link per edge
        with edge_internal == 0 in `_edges` order, as numpy arrays: edge (its index), from_unitig / from_orient (the
        unitig end it leaves: +1 its last node in listed order, -1 its first), to_unitig / to_orient (the end it
        enters: +1 the first node, -1 the last), cov.  A device graph is served by the device and stays lazy."""
        if self._on_device():
            h = self._require_device_state()
            if hasattr(h, "unitig_links"):
                return h.unitig_links()
            return self._links_over(h.arrays())
        return self._links_over(self._unitig_index_arrays())

    def read_unitig_paths(self) -> dict:
        """every read of get_reads(), in that order, as steps along the unitigs of compacted_unitigs()
        (amira_gmg_read_unitig_paths): read r's steps are path_off[r]:path_off[r + 1]; a step is a maximal run of
        consecutive windows of the read that follow one unitig, with its unitig, orient (+1: in listed order), pos
        (of its first window's node), win (that window's index in _readNodes[read]) and length (windows).  None
        windows belong to no step; short reads have empty paths.  A device graph is served by the device and stays
        lazy."""
        if self._on_device():
            h = self._require_device_state()
            if hasattr(h, "read_unitig_paths"):
                return h.read_unitig_paths()
            a = h.arrays()
            return self._read_paths_over(a, a)
        return self._read_paths_over(self._unitig_index_arrays(), self._read_index_arrays())

    def _read_index_arrays(self) -> dict:
        """the per-read window arrays _read_paths_over reads, from _readNodes / _readNodeDirections in get_reads()
        order: win_off, win_node (index in `_nodes` order, -1 for None), win_dir (0 for None); a read without an entry
        has no windows"""
        index = {nh: i for i, nh in enumerate(self._nodes)}
        rn, rd = self._readNodes, self._readNodeDirections
        nodes = [rn.get(r, []) for r in self._reads]
        dirs = [rd.get(r, []) for r in self._reads]
        node = np.asarray([index.get(x, -1) if x is not None else -1 for row in nodes for x in row], np.int64)
        return {"win_off": np.concatenate([[0], np.cumsum([len(x) for x in nodes], dtype=np.int64)]).astype(np.int64),
                "win_node": node,
                "win_dir": np.where(node >= 0, np.asarray([d or 0 for row in dirs for d in row], np.int64), 0)}

    def _links_over(self, a) -> dict:
        """amira_gmg_unitig_links over index arrays (those of _unitigs_over, and edge_cov)"""
        u = self._unitigs_over(a)
        j = np.flatnonzero(u["edge_internal"] == 0)
        src, tgt = np.asarray(a["edge_src"], np.int64)[j], np.asarray(a["edge_tgt"], np.int64)[j]
        sd, td = np.asarray(a["edge_sd"], np.int64)[j], np.asarray(a["edge_td"], np.int64)[j]
        return {"edge": j.astype(np.int32), "from_unitig": u["node_unitig"][src],
                "from_orient": (sd * u["node_orient"][src]).astype(np.int8), "to_unitig": u["node_unitig"][tgt],
                "to_orient": (td * u["node_orient"][tgt]).astype(np.int8),
                "cov": np.asarray(a["edge_cov"], np.int64)[j].astype(np.uint32)}

    def _read_paths_over(self, a, w) -> dict:
        """amira_gmg_read_unitig_paths over index arrays: the graph `a` (as _unitigs_over) and the windows `w`
        (win_off, win_node with -1 for None, win_dir).  A window continues the one before it when both are live, in
        one read, and succ(state before) == its state, a window's state being 2 * node + (dir < 0)"""
        u = self._unitigs_over(a)
        woff = np.asarray(w["win_off"], np.int64)
        node, d = np.asarray(w["win_node"], np.int64), np.asarray(w["win_dir"], np.int64)
        R, W = len(woff) - 1, len(node)
        live = node >= 0
        state = np.where(live, 2 * node + (d < 0), 0)
        cont = np.zeros(W, bool)
        if W and len(u["node_unitig"]):
            succ = self._unitig_succ(a)
            cont[1:] = live[1:] & live[:-1] & (succ[state[:-1]] == state[1:])
            cont[woff[:-1][woff[:-1] < W]] = False                # a read's first window continues nothing
        start = np.flatnonzero(live & ~cont)
        end = np.flatnonzero(live & ~np.append(cont[1:], False))
        read = np.repeat(np.arange(R, dtype=np.int64), np.diff(woff))[start]
        n = node[start]
        return {"path_off": np.concatenate([[0], np.cumsum(np.bincount(read, minlength=R))]).astype(np.int64),
                "unitig": u["node_unitig"][n], "orient": (np.where(d[start] < 0, -1, 1) * u["node_orient"][n]).astype(np.int8),
                "pos": u["node_pos"][n], "win": (start - woff[read]).astype(np.int32),
                "length": (end - start + 1).astype(np.int32)}

    def compacted_bubbles(self) -> dict:
        """the simple bubbles of the compacted graph (include/amira_gmg.h, amira_gmg_bubbles) as numpy arrays: per
        bubble its source and sink states (2 * node + side, node indices in `_nodes` order), its branches
        branch_off[b]:branch_off[b + 1]; per branch its unitig (of compacted_unitigs()), orientation (+1: entered at the
        unitig's first node) and branch_reads (the reads that run the whole branch).  A device graph is served by the
        device and stays lazy."""
        if self._on_device():
            h = self._require_device_state()
            if hasattr(h, "bubbles"):
                return h.bubbles()
            a = h.arrays()
            return self._bubbles_over(a, a)
        return self._bubbles_over(self._unitig_index_arrays(), self._read_index_arrays())

    def _bubbles_over(self, a, w) -> dict:
        """amira_gmg_bubbles over index arrays: the graph `a` (as _unitigs_over) and the windows `w` (as
        _read_paths_over).  Every directed edge is tested as a branch entry at once; the entries of the lists, in state
        order and list order, are grouped by (sigma, tau)"""
        out = {"source": np.zeros(0, np.int32), "sink": np.zeros(0, np.int32), "branch_off": np.zeros(1, np.int64),
               "branch_unitig": np.zeros(0, np.int32), "branch_orient": np.zeros(0, np.int8),
               "branch_reads": np.zeros(0, np.uint32)}
        N, E = len(a["node_cov"]), len(a["edge_src"])
        if E == 0:
            return out
        u = self._unitigs_over(a)
        src, tgt = np.asarray(a["edge_src"], np.int64), np.asarray(a["edge_tgt"], np.int64)
        sd, td = np.asarray(a["edge_sd"], np.int64), np.asarray(a["edge_td"], np.int64)
        fo, bo = np.asarray(a["fw_off"], np.int64), np.asarray(a["bw_off"], np.int64)
        size, one = self._list_sizes(a)
        nu, uoff = u["node_unitig"].astype(np.int64), u["unitig_off"]
        unodes = u["unitig_nodes"].astype(np.int64)
        listed = 2 * np.arange(N, dtype=np.int64) + (u["node_orient"] < 0)          # the state a node is listed through
        sigma, c = 2 * src + (sd < 0), 2 * tgt + (td < 0)
        b = nu[tgt]
        along = c == listed[tgt]                                                    # the walk follows b's listed order
        t = np.where(along, unodes[uoff[b + 1] - 1], unodes[uoff[b]])
        e2 = one[listed[t] ^ ~along]
        ok = (size[c ^ 1] == 1) & (u["circular"][b] == 0) & (e2 >= 0)
        e2 = np.maximum(e2, 0)
        y = tgt[e2]
        tau = 2 * y + (td[e2] < 0)
        ok &= (nu[src] != b) & (nu[y] != b) & (sigma < (tau ^ 1))
        # the list entries in state order, then list order; the branch entries grouped by (sigma, tau)
        state = np.concatenate([2 * np.repeat(np.arange(N, dtype=np.int64), np.diff(fo)),
                                2 * np.repeat(np.arange(N, dtype=np.int64), np.diff(bo)) + 1])
        ent = np.concatenate([np.asarray(a["fw_edges"], np.int64), np.asarray(a["bw_edges"], np.int64)])
        ent = ent[np.argsort(state, kind="stable")]
        ent = ent[ok[ent]]
        _, first, inv, cnt = np.unique(sigma[ent] * (2 * N) + tau[ent], return_index=True, return_inverse=True,
                                       return_counts=True)
        inv = inv.ravel()
        g = first[inv]                                                              # the entry of its group's first
        sel = np.flatnonzero(cnt[inv] >= 2)
        sel = sel[np.argsort(g[sel], kind="stable")]                                # bubble by bubble, in list order
        starts = np.flatnonzero(g[sel] == sel)
        br, heads = ent[sel], ent[sel[starts]]
        bu = nu[tgt[br]]
        p = self._read_paths_over(a, w)
        ulen = np.diff(uoff)
        branch_of = np.full(len(ulen), -1, np.int64)
        branch_of[bu] = np.arange(len(bu))
        hit = branch_of[p["unitig"]]
        full = (hit >= 0) & (p["length"] == ulen[p["unitig"]])
        out.update(source=sigma[heads].astype(np.int32), sink=tau[heads].astype(np.int32),
                   branch_off=np.append(starts, len(sel)).astype(np.int64), branch_unitig=bu.astype(np.int32),
                   branch_orient=np.where(unodes[uoff[bu]] == tgt[br], 1, -1).astype(np.int8),
                   branch_reads=np.bincount(hit[full], minlength=len(bu)).astype(np.uint32))
        return out

    def pop_compacted_bubbles(self, sample_genesOfInterest={}):
        """pop the simple bubbles of compacted_bubbles(): in each bubble keep the branch with the largest mean node
        coverage (cov_sum / length, compared exactly; ties to the most branch_reads, then to the first branch) and
        remove every other branch whole, unless one of its nodes holds a gene of sample_genesOfInterest.  Returns the
        removed node hashes in bubble order, branch order and the unitig's listed order.  Reads through a removed
        branch get None windows and are marked for correction, as with any removal.  A device graph is popped on the
        device (amira_gmg_bubbles, amira_gmg_remove_nodes) and stays lazy; a graph edited on the host is popped over
        its objects.  One call pops the bubbles present now: call again for those that popping makes."""
        if self._on_device():
            if self.get_total_number_of_nodes() == 0:
                return []
            h = self._require_device_state()
            bub, u = self.compacted_bubbles(), self.compacted_unitigs()
            (key,) = self._arrays("node_key")
            ranks = self._gene_ranks(list(sample_genesOfInterest))
            amr = np.asarray(h.nodes_containing(ranks), bool) if ranks else np.zeros(len(key), bool)
            removed = self._bubble_pop_nodes(bub, u, amr)
            if not len(removed):
                return []
            hashes = _keys.node_keys(key[removed].astype(np.int64), self._vocab)[0]
            flags = np.zeros(len(key), np.uint8)
            flags[removed] = 1
            h.remove_nodes(flags)
            self._device_ops = self._device_ops + (("remove_nodes", (flags,)),)
            self._apply_device_removal(h)
            return hashes
        nodes = self._nodes
        if not nodes:
            return []
        a = self._unitig_index_arrays()
        bub, u = self._bubbles_over(a, self._read_index_arrays()), self._unitigs_over(a)
        AMR_nodes = self.get_AMR_nodes(sample_genesOfInterest)
        order = list(nodes)
        removed = self._bubble_pop_nodes(bub, u, np.asarray([nh in AMR_nodes for nh in order], bool))
        hashes = [order[i] for i in removed.tolist()]
        for nh in hashes:
            self.remove_node(nodes[nh])
        return hashes

    @staticmethod
    def _bubble_winners(bub, u, amr) -> np.ndarray:
        """the popping policy of pop_compacted_bubbles over index arrays: bub as compacted_bubbles, u as
        compacted_unitigs, amr[n]: node n holds a gene of interest.  Returns per branch the branch of its bubble that
        is kept, or -1 for the branches that stay (the kept ones, and those with a node holding a gene of interest)."""
        off = np.asarray(bub["branch_off"], np.int64)
        d = np.diff(off)
        if not len(d):
            return np.zeros(0, np.int64)
        bu = np.asarray(bub["branch_unitig"], np.int64)
        uoff = np.asarray(u["unitig_off"], np.int64)
        ln, cs = np.diff(uoff)[bu], np.asarray(u["cov_sum"], np.int64)[bu]
        rd = np.asarray(bub["branch_reads"], np.int64)
        # every ordered pair (i, j) of branches of one bubble; i beats j on the mean coverage cs / ln (cross-multiplied),
        # then on the reads, then on the position.  The branch that beats all the others of its bubble is kept.
        pb = np.repeat(np.arange(len(d)), d * d)
        k = np.arange(len(pb)) - np.repeat(np.cumsum(d * d) - d * d, d * d)
        i, j = off[pb] + k // d[pb], off[pb] + k % d[pb]
        lhs, rhs = cs[i] * ln[j], cs[j] * ln[i]
        beats = (lhs > rhs) | ((lhs == rhs) & ((rd[i] > rd[j]) | ((rd[i] == rd[j]) & (i < j))))
        keep = np.bincount(i[beats], minlength=len(bu)) == np.repeat(d, d) - 1
        gene = np.zeros(len(uoff) - 1, bool)
        gene[np.asarray(u["node_unitig"], np.int64)[np.flatnonzero(amr)]] = True
        return np.where(~keep & ~gene[bu], np.repeat(np.flatnonzero(keep), d), -1)

    @staticmethod
    def _bubble_pop_nodes(bub, u, amr) -> np.ndarray:
        """the node indices pop_compacted_bubbles removes (the branches _bubble_winners replaces), in bubble order,
        branch order and listed order"""
        go = np.asarray(bub["branch_unitig"], np.int64)[GeneMerGraph._bubble_winners(bub, u, amr) >= 0]
        uoff = np.asarray(u["unitig_off"], np.int64)
        n = np.diff(uoff)[go]
        idx = np.repeat(uoff[go] - np.cumsum(n) + n, n) + np.arange(int(n.sum()))
        return np.asarray(u["unitig_nodes"], np.int64)[idx]

    def correct_compacted_bubbles(self, sample_genesOfInterest={}):
        """the reads rewritten through the bubbles pop_compacted_bubbles would pop (the same kept branch, the same
        branches spared for a gene of sample_genesOfInterest), as a new encode.EncodedReads to rebuild from
        (include/amira_gmg.h, amira_gmg_correct_bubble_reads): a read that runs a replaced branch whole, between the
        bubble's two junction nodes, spells the kept branch there instead; every other call is unchanged.  It shares
        the vocabulary and read ids of this graph's reads, its dicts are shallow copies with only the changed reads
        decoded, and it carries `changed` (per read) and `branch_rewritten` (per branch of compacted_bubbles()).  The
        graph and its reads are left as they are.  A device graph is corrected on the device, which writes the new CSR
        that a rebuild from the result reads without uploading it again."""
        return self._source_encoded().corrected(self._bubble_correction(sample_genesOfInterest)[0], self._device)

    def _bubble_correction(self, sample_genesOfInterest, flags_on_device=False) -> tuple:
        """correct_compacted_bubbles before it becomes an EncodedReads: (the outputs of DeviceGraph.correct_bubble_reads,
        the bubble count, the branches replaced).  A device graph whose handle has the policy is corrected on the handle
        alone (_handle_correction)."""
        src = self._source_encoded()
        if self._on_device():
            h = self._require_device_state()
            ranks = self._gene_ranks(list(sample_genesOfInterest))
            if hasattr(h, "bubble_policy"):
                return self._handle_correction(h, ranks, flags_on_device)
            bub, u = self.compacted_bubbles(), self.compacted_unitigs()
            (key,) = self._arrays("node_key")
            amr = np.asarray(h.nodes_containing(ranks), bool) if ranks else np.zeros(len(key), bool)
            rw = self._bubble_winners(bub, u, amr)
            if hasattr(h, "correct_bubble_reads"):
                out = h.correct_bubble_reads(rw, on_device=True)
            else:
                a = h.arrays()
                out = self._corrected_reads_over(u, self._read_paths_over(a, a), bub, a, key, rw, src)
            return out, len(bub["source"]), int((rw >= 0).sum())
        a, w = self._unitig_index_arrays(), self._read_index_arrays()
        u, bub = self._unitigs_over(a), self._bubbles_over(a, w)
        amr_nodes = self.get_AMR_nodes(sample_genesOfInterest)
        rank = {n: i + 1 for i, n in enumerate(src.vocab.names)}
        key = np.asarray([[g.get_strand() * rank[g.get_name()] for g in n.get_canonical_geneMer()] for n in self._nodes.values()],
                         np.int64).reshape(len(self._nodes), int(self._kmerSize))
        rw = self._bubble_winners(bub, u, np.asarray([nh in amr_nodes for nh in self._nodes], bool))
        return (self._corrected_reads_over(u, self._read_paths_over(a, w), bub, w, key, rw, src), len(bub["source"]),
                int((rw >= 0).sum()))

    @staticmethod
    def _handle_correction(h, ranks, flags_on_device) -> tuple:
        """one correction of the graph the handle holds, with the device's popping policy: the corrected CSR written on
        the device, the bubble count, the branches replaced"""
        n_replaced = h.bubble_policy(ranks)
        out = h.correct_bubble_reads(None, on_device=True, flags_on_device=flags_on_device)
        return out, h.bubble_counts()[0], n_replaced

    def correct_bubbles_until_stable(self, max_rounds=30, sample_genesOfInterest={}, filter_graph=None):
        """rounds of correct_compacted_bubbles and a rebuild from the corrected reads, until a round rewrites no read
        step or max_rounds rounds have run -> (graph, reads).  It gives exactly what this loop gives:

            cur, e = self, reads of self
            for _ in range(max_rounds):
                e2 = cur.correct_compacted_bubbles(sample_genesOfInterest)
                if not e2.branch_rewritten.any(): break
                e = e2; cur = GeneMerGraph(e, k); filter_graph and cur.filter_graph(*filter_graph)
            return cur, e

        Round 1 corrects this graph as it is (filtered, trimmed or edited on the host); every later round corrects the
        rebuild of the previous round's reads, filtered first when filter_graph = (minNodeCoverage, minEdgeCoverage).
        `graph` is lazy and owns the device handle, or is this graph when round 1 rewrites nothing.  `reads` is an
        encode.EncodedReads: `changed` is the union over the rounds, `branch_rewritten` that of the last round that
        rewrote a step, and `rounds` holds per round run (the last one included) its bubbles, branches, branches
        replaced, steps rewritten, reads rewritten and the call count after it.  This graph and its reads are left as
        they were; a device graph rebuilds its device copy when next asked for it.

        Rounds after the first run on the device handle alone: the policy, the correction and the rebuild stay on the
        GPU and only counts come back; the corrected reads are copied to the host and decoded once, at the end."""
        src = self._source_encoded()
        k = int(self._kmerSize)
        filt = None if filter_graph is None else (max(int(filter_graph[0]), 0), max(int(filter_graph[1]), 0))
        rounds, out, last, changed, filtered, h = [], None, None, None, False, None
        for r in range(max_rounds):
            if r == 0:
                x, n_bubbles, n_replaced = self._bubble_correction(sample_genesOfInterest, flags_on_device=True)
            else:
                x, n_bubbles, n_replaced = self._handle_correction(h, ranks, True)
            steps = int(x["branch_rewritten"].sum())
            rounds.append({"bubbles": n_bubbles, "branches": len(x["branch_rewritten"]), "replaced": n_replaced,
                           "steps": steps, "reads": int(x["changed"].sum()), "calls": len(x["ids"])})
            last = x
            if steps == 0:
                break
            out = x                      # the previous CSR is dropped only now, after this round's correction
            changed = x["changed"] if changed is None else _union(changed, x["changed"])
            if h is None:
                h, ranks = _handle(self._device), self._gene_ranks(list(sample_genesOfInterest))
            h.owner = None               # the graph that held the handle rebuilds on demand
            if isinstance(x["ids"], np.ndarray):
                h.build(x["ids"], x["off"], k, x["pos_start"], x["pos_end"])
            else:                        # the correction's device CSR, whose call count is known exactly
                h.build(x["ids"], x["off"], k, x["pos_start"], x["pos_end"], on_device=True, n_calls=len(x["ids"]))
            filtered = bool(filt) and h.sizes_early()["nodes"] > 0
            if filtered:
                h.filter_graph(*filt)
        if out is None:
            R = len(src.read_ids)
            reads = src.corrected({"ids": src.ids, "off": src.off, "pos_start": src.pos_start, "pos_end": src.pos_end,
                                   "changed": np.zeros(R, np.uint8),
                                   "branch_rewritten": _host(last["branch_rewritten"]) if last else np.zeros(0, np.uint32)})
            reads.rounds = rounds
            return self, reads
        reads = src.corrected({**out, "changed": _host(changed), "branch_rewritten": _host(out["branch_rewritten"])},
                              self._device)
        reads.rounds = rounds
        g = type(self)({}, self._kmerSize, device=self._device)
        g._encoded, g._reads, g._genePositions = reads, reads.reads, reads.positions
        g._adopt_build(h, reads.vocab, reads.ids, reads.off)
        if filter_graph is not None:
            g.set_minNodeCoverage(filter_graph[0])
            g.set_minEdgeCoverage(filter_graph[1])
            if filtered:
                g._device_ops = (("filter_graph", filt),)
        return g, reads

    def _source_encoded(self):
        """this graph's reads as an encode.EncodedReads: the one it was built from, or the reads encoded as the build
        encoded them"""
        if self._encoded is not None:
            return self._encoded
        e = encode.EncodedReads.__new__(encode.EncodedReads)
        e.vocab, e.ids, e.off, e.pos_start, e.pos_end = self._encode()
        e.reads, e.positions, e.read_ids, e._device = self._reads, self._genePositions or None, list(self._reads), None
        return e

    @staticmethod
    def _corrected_reads_over(u, p, bub, w, key, replace_with, src) -> dict:
        """amira_gmg_correct_bubble_reads over index arrays: u as compacted_unitigs, p as read_unitig_paths, bub as
        compacted_bubbles, the windows w (win_off, win_node with -1 for None, win_dir), node keys key[N, k], and the
        encoded reads src (ids, off, pos_start, pos_end).  Every step is tested at once; the edits (which never
        overlap) set per call its number of output calls, whose prefix sums place every call"""
        rw = np.asarray(replace_with, np.int64)
        ids, off = np.asarray(src.ids, np.int32), np.asarray(src.off, np.int64)
        ps, pe = src.pos_start, src.pos_end
        R, NB = len(off) - 1, len(rw)
        if NB:
            boff = np.asarray(bub["branch_off"], np.int64)
            of = np.repeat(np.arange(len(boff) - 1), np.diff(boff))
            bad = (rw < -1) | (rw >= NB) | (rw == np.arange(NB))
            if (bad | ((rw >= 0) & (of[np.clip(rw, 0, NB - 1)] != of))).any():
                raise ValueError("correct_bubble_reads: replace_with must hold -1 or another branch of the same bubble")
        t = np.zeros(0, np.int64)
        if NB and len(p["unitig"]):
            uoff = np.asarray(u["unitig_off"], np.int64)
            ulen = np.diff(uoff)
            bu = np.asarray(bub["branch_unitig"], np.int64)
            branch_of = np.full(len(ulen), -1, np.int64)
            branch_of[bu] = np.arange(NB)
            sun = np.asarray(p["unitig"], np.int64)
            g, m = branch_of[sun], ulen[sun]
            read = np.repeat(np.arange(R, dtype=np.int64), np.diff(p["path_off"]))
            woff = np.asarray(w["win_off"], np.int64)
            win = np.asarray(p["win"], np.int64)
            t = np.flatnonzero((g >= 0) & (rw[np.maximum(g, 0)] >= 0) & (p["length"] == m) & (win >= 1)
                               & (win + m < np.diff(woff)[read]))
            node, d = np.asarray(w["win_node"], np.int64), np.asarray(w["win_dir"], np.int64)
            before = woff[read[t]] + win[t] - 1
            after = before + m[t] + 1
            sp, sn = 2 * node[before] + (d[before] < 0), 2 * node[after] + (d[after] < 0)
            q = of[g[t]]
            sigma, tau = np.asarray(bub["source"], np.int64)[q], np.asarray(bub["sink"], np.int64)[q]
            fwd = (sp == sigma) & (sn == tau)
            ok = (node[before] >= 0) & (node[after] >= 0) & (fwd | ((sp == tau ^ 1) & (sn == sigma ^ 1)))
            t, fwd = t[ok], fwd[ok]
        changed = np.zeros(R, np.uint8)
        rewritten = np.zeros(NB, np.uint32)
        count = np.ones(len(ids), np.int64)
        touched = np.zeros(len(ids), bool)
        if len(t):
            r, gt, mt = read[t], g[t], m[t]
            keep = rw[gt]
            kb = bu[keep]
            m2 = ulen[kb]
            c0 = off[r] + win[t]
            rep = np.repeat(c0 - np.cumsum(mt) + mt, mt) + np.arange(int(mt.sum()))
            touched[rep] = True
            count[rep] = 0
            count[c0] = m2
            changed[r] = 1
            rewritten = np.bincount(gt, minlength=NB).astype(np.uint32)
        idx = np.concatenate([[0], np.cumsum(count)]).astype(np.int64)
        total = int(idx[-1])
        out = {"ids": np.empty(total, np.int32), "off": idx[off],
               "pos_start": None if ps is None else np.empty(total, np.int32),
               "pos_end": None if pe is None else np.empty(total, np.int32), "changed": changed, "branch_rewritten": rewritten}
        keep_calls = np.flatnonzero(~touched)
        out["ids"][idx[keep_calls]] = ids[keep_calls]
        for f, x in (("pos_start", ps), ("pos_end", pe)):
            if x is not None:
                out[f][idx[keep_calls]] = x[keep_calls]
        if len(t):
            e = np.repeat(np.arange(len(t)), m2)
            j = np.arange(int(m2.sum())) - np.repeat(np.cumsum(m2) - m2, m2)
            walk = np.where(fwd, 1, -1)[e] * np.asarray(bub["branch_orient"], np.int64)[keep[e]]
            n = np.asarray(u["unitig_nodes"], np.int64)[np.where(walk > 0, uoff[kb[e]] + j, uoff[kb[e]] + m2[e] - 1 - j)]
            key = np.asarray(key, np.int64)
            out["ids"][idx[c0[e]] + j] = np.where(walk * np.asarray(u["node_orient"], np.int64)[n] > 0, key[n, 0], -key[n, -1])
            for f, x in (("pos_start", ps), ("pos_end", pe)):
                if x is not None:
                    out[f][idx[c0[e]] + j] = x[c0[e] + np.minimum(j, mt[e] - 1)]
        return out

    def _on_device(self) -> bool:
        """the device copy still is this graph (no host-side mutation since the build / last device operation)"""
        return bool(self._device_synced) and len(self._reads) > 0

    def get_total_number_of_nodes(self) -> int:
        if self.__dict__.get("_lazy"):
            return self._require_device_state().sizes_early()["nodes"]
        return len(self._nodes)

    def get_total_number_of_edges(self) -> int:
        if self.__dict__.get("_lazy"):
            return self._require_device_state().sizes_early()["edges"]
        return len(self._edges)

    def get_total_number_of_reads(self) -> int:
        return len(self._reads)

    def get_degree(self, node) -> int:
        return len(node.get_forward_edge_hashes()) + len(node.get_backward_edge_hashes())

    def get_forward_edges(self, node):
        return [self._edges[h] for h in node.get_forward_edge_hashes()]

    def get_backward_edges(self, node):
        return [self._edges[h] for h in node.get_backward_edge_hashes()]

    def get_forward_neighbors(self, node):
        return [e.get_targetNode() for e in self.get_forward_edges(node)]

    def get_backward_neighbors(self, node):
        return [e.get_targetNode() for e in self.get_backward_edges(node)]

    def get_all_neighbors(self, node):
        return self.get_forward_neighbors(node) + self.get_backward_neighbors(node)

    def get_all_neighbor_hashes(self, node) -> set:
        return {n.__hash__() for n in self.get_all_neighbors(node)}

    def check_if_nodes_are_adjacent(self, sourceNode, targetNode) -> bool:
        return (targetNode.__hash__() in self.get_all_neighbor_hashes(sourceNode)
                and sourceNode.__hash__() in self.get_all_neighbor_hashes(targetNode))

    def get_edge_hashes_between_nodes(self, sourceNode, targetNode):
        assert self.check_if_nodes_are_adjacent(sourceNode, targetNode)
        out = [e.__hash__() for e in self.get_forward_edges(sourceNode) + self.get_backward_edges(sourceNode)
               if e.get_targetNode() == targetNode]
        back = [e.__hash__() for e in self.get_forward_edges(targetNode) + self.get_backward_edges(targetNode)
                if e.get_targetNode() == sourceNode]
        if len(out) > 1 or len(back) > 1:
            return (out, back)
        return (out[0], back[0])

    def get_edges_between_nodes(self, sourceNode, targetNode):
        s2t, t2s = self.get_edge_hashes_between_nodes(sourceNode, targetNode)
        if isinstance(s2t, list) or isinstance(t2s, list):
            return [self._edges[h] for h in s2t], [self._edges[h] for h in t2s]
        return self._edges[s2t], self._edges[t2s]

    def remove_junk_reads(self, error_rate):
        """upstream construct_graph.py:1398-1420: reads with more than round(n * (1 - error_rate)) filtered
        (None) nodes are rejected.  On the device: one thread per read counts its None windows (k_junk_read_mask)."""
        reads, positions = self._reads, self._genePositions
        kept, kept_pos, rejected, rejected_pos = {}, {}, {}, {}
        if self._on_device():
            mask = self._require_device_state().junk_read_mask(error_rate).tolist()
            for read_id, m in zip(self._read_ids, mask):
                if m == 2:
                    continue             # short read: not in _readNodes
                (kept if m else rejected)[read_id] = reads[read_id]
                (kept_pos if m else rejected_pos)[read_id] = positions[read_id]
            return kept, kept_pos, rejected, rejected_pos
        for read_id, nodes in self._readNodes.items():
            ok = nodes.count(None) <= round(len(nodes) * (1 - error_rate))
            (kept if ok else rejected)[read_id] = reads[read_id]
            (kept_pos if ok else rejected_pos)[read_id] = positions[read_id]
        return kept, kept_pos, rejected, rejected_pos

    def get_valid_reads_only(self):
        """upstream construct_graph.py:1422-1427"""
        if self.__dict__.get("_lazy"):
            to_correct = self._arrays("to_correct")[0].tolist()
            return {r: self._reads[r] for r, bad in zip(self._read_ids, to_correct) if not bad}
        bad = self._readsToCorrect
        return {r: calls for r, calls in self._reads.items() if r not in bad}

    def get_all_node_coverages(self):
        if self.__dict__.get("_lazy"):
            return self._arrays("node_cov")[0].tolist()
        return [n.get_node_coverage() for n in self._nodes.values()]

    def get_mean_node_coverage(self):
        """upstream construct_graph.py:868-871 (statistics.mean of the coverages: exact, int when it divides)"""
        if self._on_device():
            n = self.get_total_number_of_nodes()
            if n == 0:
                raise statistics.StatisticsError("mean requires at least one data point")
            total, _ = self._require_device_state().node_coverage_stats()
            return total // n if total % n == 0 else total / n
        return statistics.mean(self.get_all_node_coverages())

    # ------------------------------------------------------------------ single-object mutators (host)
    def _touch(self):
        self._nodes                          # host edits need the host objects (materialise before going stale)
        self._device_synced = False
        self._index_cache = None

    def add_node_to_read(self, node, readId: str, node_direction: int, node_position=None):
        self._touch()
        if readId not in self._readNodes:
            self._readNodes[readId] = []
            self._readNodeDirections[readId] = []
            self._readNodePositions[readId] = []
        self._readNodes[readId].append(node.__hash__())
        self._readNodeDirections[readId].append(node_direction)
        self._readNodePositions[readId].append(node_position)
        return self._readNodes[readId]

    def add_node_to_nodes(self, node, nodeHash: int) -> None:
        self._touch()
        self._nodes[nodeHash] = node

    def add_node(self, geneMer, reads: list):
        self._touch()
        nodeHash = geneMer.__hash__()
        node = self._nodes.get(nodeHash)
        if node is None:
            node = self._cls.Node(geneMer)
            self._nodes[nodeHash] = node
        for r in reads:
            node.add_read(r)
        return node

    def create_edges(self, sourceNode, targetNode, sourceGeneMerDirection: int, targetGeneMerDirection: int):
        E = self._cls.Edge
        return (E(sourceNode, targetNode, sourceGeneMerDirection, targetGeneMerDirection),
                E(targetNode, sourceNode, targetGeneMerDirection * -1, sourceGeneMerDirection * -1))

    def add_edge_to_edges(self, edge):
        self._touch()
        return self._edges.setdefault(edge.__hash__(), edge)

    def add_edges_to_graph(self, sourceToTargetEdge, reverseTargetToSourceEdge):
        return self.add_edge_to_edges(sourceToTargetEdge), self.add_edge_to_edges(reverseTargetToSourceEdge)

    def add_edge_to_node(self, node, edge):
        self._touch()
        if edge.get_sourceNodeDirection() == 1:
            node.add_forward_edge_hash(edge.__hash__())
        if edge.get_sourceNodeDirection() == -1:
            node.add_backward_edge_hash(edge.__hash__())
        return node

    def add_edge(self, sourceGeneMer, targetGeneMer):
        sourceNode = self.add_node(sourceGeneMer, [])
        targetNode = self.add_node(targetGeneMer, [])
        fwd, rev = self.create_edges(sourceNode, targetNode, sourceGeneMer.get_geneMerDirection(),
                                     targetGeneMer.get_geneMerDirection())
        fwd, rev = self.add_edges_to_graph(fwd, rev)
        self.add_edge_to_node(sourceNode, fwd)
        self.add_edge_to_node(targetNode, rev)
        return fwd, rev

    def remove_edge_from_edges(self, edgeHash: int) -> None:
        self._touch()
        del self._edges[edgeHash]
        assert edgeHash not in self._edges, "This edge was not removed from the graph successfully"

    def remove_edge(self, edgeHash: int) -> None:
        edge = self._edges.get(edgeHash)
        if edge is None:
            return
        self._touch()
        if edge.get_sourceNodeDirection() == 1:
            edge.get_sourceNode().remove_forward_edge_hash(edgeHash)
        if edge.get_sourceNodeDirection() == -1:
            edge.get_sourceNode().remove_backward_edge_hash(edgeHash)
        del self._edges[edgeHash]

    def remove_node_from_reads(self, node_to_remove) -> None:
        self._touch()
        gone = node_to_remove.__hash__()
        for readId in node_to_remove.get_reads():
            keep = [h != gone for h in self._readNodes[readId]]
            for table in (self._readNodes, self._readNodeDirections, self._readNodePositions):
                table[readId] = [v if kp else None for v, kp in zip(table[readId], keep)]
            self._readsToCorrect.add(readId)

    def remove_node(self, node):
        nodeHash = node.__hash__()
        assert nodeHash in self._nodes, "This node is not in the graph"
        assert node == self._nodes[nodeHash]
        self.remove_node_from_reads(node)
        for edgeHash in set(node.get_forward_edge_hashes() + node.get_backward_edge_hashes()):
            targetNode = self._edges[edgeHash].get_targetNode()
            for e in self.get_edge_hashes_between_nodes(node, targetNode):
                self.remove_edge(e)
        del self._nodes[nodeHash]

    def set_minNodeCoverage(self, minNodeCoverage: int):
        self._minNodeCoverage = minNodeCoverage
        return self._minNodeCoverage

    def set_minEdgeCoverage(self, minEdgeCoverage: int):
        self._minEdgeCoverage = minEdgeCoverage
        return self._minEdgeCoverage

    def list_nodes_to_remove(self, minNodeCoverage: int):
        return {n for n in self._nodes.values() if not n.get_node_coverage() > minNodeCoverage - 1}

    def list_edges_to_remove(self, minEdgeCoverage: int, nodesToRemove):
        doomed = set()
        for eh, e in self._edges.items():
            if not e.get_edge_coverage() > minEdgeCoverage - 1:
                doomed.add(eh)
            if e.get_sourceNode() in nodesToRemove or e.get_targetNode() in nodesToRemove:
                doomed.add(eh)
        return doomed

    # ------------------------------------------------------------------ components
    def dfs_component(self, start, component_id, visited=None):
        if visited is None:
            visited = set()
        stack = [start]
        visited.add(start.__hash__())
        while stack:
            node = stack.pop()
            node.set_component(component_id)
            for nb in self.get_all_neighbors(node):
                if nb.__hash__() not in visited:
                    visited.add(nb.__hash__())
                    stack.append(nb)

    def assign_component_ids(self):
        """component ids 1, 2, ... in order of each component's first node (upstream :920-927)"""
        visited = set()
        component_id = 1
        for nodeHash, node in self._nodes.items():
            if nodeHash not in visited:
                self.dfs_component(node, component_id, visited)
                component_id += 1

    def get_nodes_in_component(self, component):
        return [n for n in self._nodes.values() if n.get_component() == int(component)]

    def components(self) -> list:
        if self.__dict__.get("_lazy"):
            return sorted(set(self._arrays("node_comp")[0].tolist()))
        return sorted({n.get_component() for n in self._nodes.values()})

    def get_number_of_component(self) -> int:
        return len(self.components())

    # ------------------------------------------------------------------ GML (upstream :542-654, 873-909)
    def write_node_entry(self, node_id, node_string, node_coverage, reads, component_ID, nodeColor):
        lines = ["\tnode\t[", "\t\tid\t%s" % node_id, '\t\tlabel\t"%s"' % node_string,
                 "\t\tcoverage\t%s" % node_coverage]
        if component_ID:
            lines.append("\t\tcomponent\t%s" % component_ID)
        lines.append('\t\treads\t"%s"' % ",".join(reads))
        if nodeColor:
            lines.append('\t\tcolor\t"%s"' % nodeColor)
        lines.append("\t]")
        return "\n".join(lines)

    def write_edge_entry(self, source_node, target_node, source_edge_direction, target_edge_direction, edge_coverage):
        return "\n".join(["\tedge\t[", "\t\tsource\t%s" % source_node, "\t\ttarget\t%s" % target_node,
                          "\t\tsource_direction\t%s" % source_edge_direction,
                          "\t\ttarget_direction\t%s" % target_edge_direction,
                          "\t\tweight\t%s" % edge_coverage, "\t]"])

    def assign_Id_to_nodes(self):
        for i, node in enumerate(self._nodes.values()):
            assert node.assign_node_Id(i) == i, "This node was assigned an incorrect ID"

    def write_gml_to_file(self, output_file, gml_content):
        d = os.path.dirname(output_file)
        if d != "" and not os.path.exists(d):
            os.mkdir(d)
        with open(output_file + ".gml", "w") as f:
            f.write("\n".join(gml_content))

    def get_gene_mer_genes(self, sourceNode) -> list:
        return [convert_int_strand_to_string(g.get_strand()) + g.get_name() for g in sourceNode.get_canonical_geneMer()]

    def get_reverse_gene_mer_genes(self, sourceNode) -> list:
        return [convert_int_strand_to_string(g.get_strand()) + g.get_name() for g in sourceNode.get_reverse_geneMer()]

    def get_gene_mer_label(self, sourceNode) -> str:
        return "~~~".join(self.get_gene_mer_genes(sourceNode))

    def _gml_from_arrays(self) -> list:
        """the GML entries of upstream generate_gml (construct_graph.py:873-909) straight from the device arrays: node id =
        insertion index, label from the canonical gene-mer, reads by id, edges in forward-then-backward list order"""
        a = self._arrays()
        names = self._vocab.names
        signed = [None] * (2 * len(names) + 1)
        V = len(names)
        for r, n in enumerate(names, 1):
            signed[V + r], signed[V - r] = "+" + n, "-" + n
        key = (a["node_key"].astype(np.int64) + V).tolist()
        cov, comp = a["node_cov"].tolist(), a["node_comp"].tolist()
        roff, reads = a["node_reads_off"].tolist(), a["node_reads"].tolist()
        fo, fe, bo, be = a["fw_off"].tolist(), a["fw_edges"].tolist(), a["bw_off"].tolist(), a["bw_edges"].tolist()
        tgt, sd, td, ecov = a["edge_tgt"].tolist(), a["edge_sd"].tolist(), a["edge_td"].tolist(), a["edge_cov"].tolist()
        rid = self._read_ids
        out = ["graph\t[", "multigraph 1"]
        for i in range(len(cov)):
            out.append(self.write_node_entry(i, "~~~".join(signed[g] for g in key[i]), cov[i],
                                             [rid[r] for r in reads[roff[i]:roff[i + 1]]], comp[i], None))
            for e in fe[fo[i]:fo[i + 1]] + be[bo[i]:bo[i + 1]]:
                if ecov[e] == 0:
                    continue
                out.append(self.write_edge_entry(i, tgt[e], sd[e], td[e], ecov[e]))
        out.append("]")
        return out

    def generate_gml(self, output_file: str, geneMerSize: int, min_node_coverage: int, min_edge_coverage: int):
        if self.__dict__.get("_lazy") or (self._on_device() and not any(n.get_color() for n in self._node_objs)):
            graph_data = self._gml_from_arrays()
            if not self.__dict__.get("_lazy"):
                self.assign_Id_to_nodes()
            self.write_gml_to_file(".".join([output_file, str(geneMerSize), str(min_node_coverage), str(min_edge_coverage)]),
                                   graph_data)
            return graph_data
        graph_data = ["graph\t[", "multigraph 1"]
        self.assign_Id_to_nodes()
        for node in self._nodes.values():
            graph_data.append(self.write_node_entry(node.get_node_Id(), self.get_gene_mer_label(node),
                                                    node.get_node_coverage(), list(node.get_reads()),
                                                    node.get_component(), node.get_color()))
            for edge in self.get_forward_edges(node) + self.get_backward_edges(node):
                if edge.get_edge_coverage() == 0:
                    continue
                graph_data.append(self.write_edge_entry(node.get_node_Id(), edge.get_targetNode().get_node_Id(),
                                                        edge.get_sourceNodeDirection(), edge.get_targetNodeDirection(),
                                                        edge.get_edge_coverage()))
        graph_data.append("]")
        self.write_gml_to_file(".".join([output_file, str(geneMerSize), str(min_node_coverage), str(min_edge_coverage)]),
                               graph_data)
        return graph_data


def bind_upstream(upstream_construct_graph):
    """Subclass upstream's own GeneMerGraph so that every correction / path-finding method it defines
    runs unchanged on a graph built by the CUDA path.

        import amira.construct_graph as cg
        import amira_b200
        cg.GeneMerGraph = amira_b200.bind_upstream(cg)       # before amira.graph_utils is imported

    The element objects are upstream's own Gene / GeneMer / Node / Edge classes."""
    up = upstream_construct_graph
    import importlib
    gene_mod = importlib.import_module(up.GeneMer.__module__.rsplit(".", 1)[0] + ".construct_gene")
    UpGene, UpGeneMer, UpNode, UpEdge = gene_mod.Gene, up.GeneMer, up.Node, up.Edge

    class _Up:
        Gene, GeneMer, Node, Edge = UpGene, UpGeneMer, UpNode, UpEdge

        @staticmethod
        def make_gene(name, strand):
            g = object.__new__(UpGene)
            g.name, g.strand = name, strand
            return g

        @staticmethod
        def make_genemer(canonical, rc, direction, node_hash):
            gm = object.__new__(UpGeneMer)
            gm.canonicalGeneMer, gm.rcGeneMer = canonical, rc
            gm.geneMerSize = len(canonical)
            gm.geneMerDirection = direction
            return gm

        @staticmethod
        def make_node(genemer, node_hash, cov, reads, comp):
            n = object.__new__(UpNode)
            n.geneMer = genemer
            n.canonicalGeneMer = genemer.canonicalGeneMer
            n.reverseGeneMer = genemer.rcGeneMer
            n.geneMerHash = node_hash
            n.nodeCoverage = cov
            n.listOfReads = reads
            n.forwardEdgeHashes = []
            n.backwardEdgeHashes = []
            n._color = None
            n._component_ID = comp
            return n

        @staticmethod
        def make_edge(src, tgt, sd, td, cov):
            e = UpEdge(src, tgt, sd, td)
            e.edgeCoverage = cov
            return e

    ours = GeneMerGraph
    gpu_methods = ("__init__", "_encode", "_build_on_device", "_materialise", "_materialise_now", "_arrays", "_on_device",
                   "_require_device_state", "_apply_device_removal", "filter_graph", "remove_low_coverage_components",
                   "_touch", "remove_junk_reads", "get_valid_reads_only", "get_total_number_of_nodes",
                   "get_total_number_of_edges", "get_all_node_coverages", "get_mean_node_coverage", "components",
                   "get_nodes_containing", "_gene_ranks", "get_AMR_nodes", "remove_non_AMR_associated_nodes", "_linear_steps",
                   "_walk", "_walks_over", "_device_walks", "_device_walk", "_short_path_nodes", "get_forward_path_from_node", "get_backward_path_from_node", "get_linear_path_for_node",
                   "remove_short_linear_paths", "compacted_unitigs", "_unitig_index_arrays", "_unitigs_over",
                   "_unitig_succ", "compacted_links", "read_unitig_paths", "_read_index_arrays", "_links_over",
                   "_read_paths_over", "_list_sizes", "compacted_bubbles", "_bubbles_over", "pop_compacted_bubbles",
                   "_bubble_pop_nodes", "_bubble_winners", "correct_compacted_bubbles", "_source_encoded",
                   "_corrected_reads_over", "_adopt_build", "_bubble_correction", "_handle_correction",
                   "correct_bubbles_until_stable",
                   "_gml_from_arrays", "generate_gml") + _LAZY_ATTRS
    ns = {name: ours.__dict__[name] for name in gpu_methods}
    ns["_cls"] = _Up
    # host mutators must mark the device copy stale
    for name in ("add_node", "add_node_to_read", "add_node_to_nodes", "add_edge_to_edges", "add_edge_to_node",
                 "remove_edge", "remove_edge_from_edges", "remove_node_from_reads"):
        base = getattr(up.GeneMerGraph, name)

        def wrapped(self, *a, _base=base, **kw):
            self._nodes                      # host edits need the host objects
            self._device_synced = False
            return _base(self, *a, **kw)

        wrapped.__name__ = name
        ns[name] = wrapped
    return type("GeneMerGraph", (up.GeneMerGraph,), ns)
