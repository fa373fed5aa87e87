"""Thin object over the C-ABI handle: integer CSR in, graph arrays out.

This is the level the parity tests and bench.py drive: it makes exactly the calls a maintainer's
ctypes stub would make (INTEGRATION.md) and returns the exported arrays unchanged."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


# the arrays of amira_gmg_unitigs, in its argument order
UNITIG_FIELDS = ("node_unitig", "node_pos", "node_orient", "unitig_off", "unitig_nodes", "circular", "cov_sum", "cov_min",
                 "cov_max", "edge_internal")
# the arrays of amira_gmg_unitig_links and amira_gmg_read_unitig_paths, in their argument order
LINK_FIELDS = ("edge", "from_unitig", "from_orient", "to_unitig", "to_orient", "cov")
PATH_FIELDS = ("path_off", "unitig", "orient", "pos", "win", "length")
# the arrays of amira_gmg_bubbles, in its argument order
BUBBLE_FIELDS = ("source", "sink", "branch_off", "branch_unitig", "branch_orient", "branch_reads")
# the arrays of amira_gmg_tips, in its argument order
TIP_FIELDS = ("tip_unitig", "tip_orient", "tip_attach", "tip_reads")
# the arrays of amira_gmg_gene_paths, in its argument order, with their types
GENE_PATH_FIELDS = (("occ_read", np.int32), ("occ_win", np.int32), ("occ_length", np.int32), ("occ_flanks", np.uint8),
                    ("occ_orient", np.int8), ("occ_cluster", np.int32), ("key_off", np.int64), ("key_state", np.int32),
                    ("n_complete", np.uint32), ("member_off", np.int64), ("members", np.int32))


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if hasattr(a, "data_ptr"):      # torch tensor (host pinned or device)
        return C.c_void_p(a.data_ptr())
    return C.c_void_p(int(a))


class DeviceGraph:
    """one GeneMerGraph build resident on one GPU"""

    def __init__(self, device: int = 0, stream: int | None = None, profiling: bool = False):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        _lib.check(self._lib.amira_gmg_create(C.byref(self._h), int(device), C.c_void_p(stream) if stream else None))
        self.device = device
        self.k = None
        self.R = 0
        self.has_pos = False
        self._keep = None
        if profiling:
            self.set_profiling(True)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.amira_gmg_destroy(self._h)
            self._h = None

    __del__ = close

    def set_profiling(self, on: bool):
        _lib.check(self._lib.amira_gmg_set_profiling(self._h, int(on)))

    def reserve(self, n_nodes: int, n_edges: int):
        _lib.check(self._lib.amira_gmg_reserve(self._h, int(n_nodes), int(n_edges)))

    def build(self, ids, off, k: int, pos_start=None, pos_end=None, on_device: bool = False, wait: bool = True,
              n_calls: int | None = None):
        """amira_gmg_build; ids/off are numpy arrays, torch tensors or raw pointers.  n_calls: the call count off[R] of a
        device CSR, when the caller knows it (amira_gmg_input_calls): the build then copies nothing back to size itself.

        The library only enqueues the build; problems the device finds (a palindromic gene-mer, a table that
        has to grow) surface at the first call that needs a result.  wait=True (default) asks for the early
        sizes right away so that they surface here, as upstream's constructor raises; wait=False returns
        as soon as the build is enqueued."""
        if isinstance(ids, np.ndarray):
            ids = np.ascontiguousarray(ids, np.int32)
            off = np.ascontiguousarray(off, np.int64)
            if pos_start is not None:
                pos_start = np.ascontiguousarray(pos_start, np.int32)
                pos_end = np.ascontiguousarray(pos_end, np.int32)
        R = (off.shape[0] if hasattr(off, "shape") else len(off)) - 1
        self._keep = (ids, off, pos_start, pos_end)   # borrowed by the library until the next build
        self.k, self.R, self.has_pos = int(k), int(R), pos_start is not None
        if on_device and n_calls is not None and R > 0:
            _lib.check(self._lib.amira_gmg_input_calls(self._h, _ptr(off), R, int(n_calls)))
        _lib.check(self._lib.amira_gmg_build(self._h, _ptr(ids), _ptr(off), R, int(k), _ptr(pos_start), _ptr(pos_end),
                                             int(on_device)))
        if wait:
            self.sizes_early()
        return self

    def build_resident(self, encoded, k: int, device: int | None = None):
        """build from an encode.EncodedReads whose CSR stays on the GPU between builds (k sweeps, rebuilds); its host
        CSR gives the call count, so the build copies nothing back to size itself"""
        ids, off, ps, pe = encoded.device_csr(self.device if device is None else device)
        return self.build(ids, off, k, ps, pe, on_device=True, n_calls=len(encoded.ids))

    def sync(self):
        _lib.check(self._lib.amira_gmg_sync(self._h))

    def filter_graph(self, min_node_cov: int, min_edge_cov: int):
        _lib.check(self._lib.amira_gmg_filter(self._h, int(min_node_cov), int(min_edge_cov)))
        return self

    def remove_low_coverage_components(self, min_component_cov: int):
        _lib.check(self._lib.amira_gmg_remove_low_coverage_components(self._h, int(min_component_cov)))

    # ---- post-build scans on the device-resident graph (include/amira_gmg.h, SURVEY.md 8f) ----------
    def read_length_coverages(self, min_lens) -> np.ndarray:
        """sums[i] = number of (node, read) incidences whose read has >= min_lens[i] gene calls"""
        ml = np.ascontiguousarray(min_lens, np.int32)
        out = np.zeros(len(ml), np.int64)
        _lib.check(self._lib.amira_gmg_read_length_coverages(self._h, _ptr(ml), len(ml), _ptr(out)))
        return out

    def node_coverage_stats(self):
        s, m = C.c_int64(), C.c_uint32()
        _lib.check(self._lib.amira_gmg_node_coverage_stats(self._h, C.byref(s), C.byref(m)))
        return s.value, m.value

    def junk_read_mask(self, error_rate: float) -> np.ndarray:
        """1 = kept, 0 = rejected, 2 = short read (upstream remove_junk_reads)"""
        mask = np.zeros(self.R, np.uint8)
        _lib.check(self._lib.amira_gmg_junk_read_mask(self._h, float(error_rate), _ptr(mask)))
        return mask

    def nodes_containing(self, ranks) -> np.ndarray:
        r = np.ascontiguousarray(ranks, np.int32)
        flags = np.zeros(self.sizes_early()["nodes"], np.uint8)
        _lib.check(self._lib.amira_gmg_nodes_containing(self._h, _ptr(r), len(r), _ptr(flags)))
        return flags.astype(bool)

    def remove_nodes(self, remove_flags):
        f = np.ascontiguousarray(remove_flags, np.uint8)
        assert len(f) == self.sizes_early()["nodes"]
        _lib.check(self._lib.amira_gmg_remove_nodes(self._h, _ptr(f)))

    def remove_nodes_without_reads_of(self, ranks):
        r = np.ascontiguousarray(ranks, np.int32)
        _lib.check(self._lib.amira_gmg_remove_nodes_without_reads_of(self._h, _ptr(r), len(r)))

    def linear_steps(self) -> dict:
        n = self.sizes()["nodes"]
        a = {"degree": np.zeros(n, np.uint32), "fw_next": np.zeros(n, np.int32), "fw_dir": np.zeros(n, np.int8),
             "fw_ext": np.zeros(n, np.uint8), "bw_next": np.zeros(n, np.int32), "bw_dir": np.zeros(n, np.int8),
             "bw_ext": np.zeros(n, np.uint8)}
        _lib.check(self._lib.amira_gmg_linear_steps(self._h, *[_ptr(a[f]) for f in ("degree", "fw_next", "fw_dir", "fw_ext",
                                                                                     "bw_next", "bw_dir", "bw_ext")]))
        return a

    def linear_walks(self, states, want_branched: bool = False):
        """walks from the states 2 * node + side (0 = forward list, 1 = backward list), without the start node, plus the
        branching node when want_branched -> (off[n + 1] int64, nodes int32): walk i is nodes[off[i]:off[i + 1]]"""
        s = np.asarray(states, np.int64).ravel()
        if len(s) and (s.min() < -2**31 or s.max() >= 2**31):
            raise ValueError("linear_walks: state out of range")
        s = np.ascontiguousarray(s, np.int32)
        off = np.zeros(len(s) + 1, np.int64)
        _lib.check(self._lib.amira_gmg_linear_walks(self._h, _ptr(s), len(s), int(bool(want_branched)), _ptr(off), None))
        nodes = np.empty(int(off[-1]), np.int32)
        if len(nodes):
            _lib.check(self._lib.amira_gmg_linear_walks(self._h, _ptr(s), len(s), int(bool(want_branched)), _ptr(off),
                                                        _ptr(nodes)))
        return off, nodes

    def unitigs(self) -> dict:
        """the compacted graph (amira_gmg_unitigs): per node its unitig, position and orientation; per unitig its
        nodes (unitig_nodes[unitig_off[u]:unitig_off[u + 1]]), circular flag and coverage sum / min / max; per directed
        edge whether it joins consecutive nodes of one unitig"""
        U = C.c_int64()
        _lib.check(self._lib.amira_gmg_unitigs(self._h, C.byref(U), *[None] * 10))
        s = self.sizes_early()
        n, m, U = s["nodes"], s["edges"], U.value
        a = {"node_unitig": np.empty(n, np.int32), "node_pos": np.empty(n, np.int32), "node_orient": np.empty(n, np.int8),
             "unitig_off": np.empty(U + 1, np.int64), "unitig_nodes": np.empty(n, np.int32),
             "circular": np.empty(U, np.uint8), "cov_sum": np.empty(U, np.int64), "cov_min": np.empty(U, np.uint32),
             "cov_max": np.empty(U, np.uint32), "edge_internal": np.empty(m, np.uint8)}
        _lib.check(self._lib.amira_gmg_unitigs(self._h, None, *[_ptr(a[f]) for f in UNITIG_FIELDS]))
        return a

    def unitig_links(self) -> dict:
        """the junction edges of the compacted graph (amira_gmg_unitig_links), in edge order: per link its edge index,
        the unitig and orientation it leaves and enters (+1: in the unitig's listed order), and the edge's coverage"""
        L = C.c_int64()
        _lib.check(self._lib.amira_gmg_unitig_links(self._h, C.byref(L), *[None] * 6))
        L = L.value
        a = {"edge": np.empty(L, np.int32), "from_unitig": np.empty(L, np.int32), "from_orient": np.empty(L, np.int8),
             "to_unitig": np.empty(L, np.int32), "to_orient": np.empty(L, np.int8), "cov": np.empty(L, np.uint32)}
        _lib.check(self._lib.amira_gmg_unitig_links(self._h, None, *[_ptr(a[f]) for f in LINK_FIELDS]))
        return a

    def read_unitig_paths(self) -> dict:
        """every read as steps along the unitigs (amira_gmg_read_unitig_paths): read r's steps are
        path_off[r]:path_off[r + 1]; per step its unitig, orientation, position of its first window, that window's
        index within the read, and its number of windows"""
        off = np.zeros(self.R + 1, np.int64)
        _lib.check(self._lib.amira_gmg_read_unitig_paths(self._h, _ptr(off), *[None] * 5))
        T = int(off[-1])
        a = {"path_off": off, "unitig": np.empty(T, np.int32), "orient": np.empty(T, np.int8), "pos": np.empty(T, np.int32),
             "win": np.empty(T, np.int32), "length": np.empty(T, np.int32)}
        _lib.check(self._lib.amira_gmg_read_unitig_paths(self._h, *[_ptr(a[f]) for f in PATH_FIELDS]))
        return a

    def bubbles(self) -> dict:
        """the simple bubbles of the compacted graph (amira_gmg_bubbles): per bubble its source and sink states, its
        branches branch_off[b]:branch_off[b + 1]; per branch its unitig, orientation (+1: entered at the unitig's first
        node) and the number of reads that run the whole branch"""
        B, NB = C.c_int64(), C.c_int64()
        _lib.check(self._lib.amira_gmg_bubbles(self._h, C.byref(B), C.byref(NB), *[None] * 6))
        B, NB = B.value, NB.value
        a = {"source": np.empty(B, np.int32), "sink": np.empty(B, np.int32), "branch_off": np.zeros(B + 1, np.int64),
             "branch_unitig": np.empty(NB, np.int32), "branch_orient": np.empty(NB, np.int8),
             "branch_reads": np.empty(NB, np.uint32)}
        _lib.check(self._lib.amira_gmg_bubbles(self._h, None, None, *[_ptr(a[f]) for f in BUBBLE_FIELDS]))
        return a

    def bubble_counts(self) -> tuple:
        """(bubbles, branches) of bubbles(), without exporting them"""
        B, NB = C.c_int64(), C.c_int64()
        _lib.check(self._lib.amira_gmg_bubbles(self._h, C.byref(B), C.byref(NB), *[None] * 6))
        return B.value, NB.value

    def bubble_policy(self, spare_ranks=(), want_replace_with: bool = False):
        """the popping policy over bubbles() (amira_gmg_bubble_policy): per bubble the branch with the largest mean node
        coverage (then most branch_reads, then the first) replaces every other branch without a node holding one of the
        genes of spare_ranks (vocabulary ranks).  Returns the number of branches replaced, and with want_replace_with
        also replace_with (per branch: its replacement, or -1) as a numpy array.  The device keeps replace_with for
        correct_bubble_reads(None)."""
        r = np.ascontiguousarray(spare_ranks, np.int32)
        n = C.c_int64()
        _lib.check(self._lib.amira_gmg_bubble_policy(self._h, _ptr(r), len(r), C.byref(n), None))
        if not want_replace_with:
            return n.value
        rw = np.empty(self.bubble_counts()[1], np.int32)
        if len(rw):
            _lib.check(self._lib.amira_gmg_bubble_policy(self._h, _ptr(r), len(r), None, _ptr(rw)))
        return n.value, rw

    def correct_bubble_reads(self, replace_with=None, on_device: bool = False, flags_on_device: bool = False) -> dict:
        """the reads through the bubbles of bubbles() rewritten along a kept branch (amira_gmg_correct_bubble_reads):
        replace_with[g] = -1 leaves branch g's reads alone, otherwise it is the branch of the same bubble whose genes
        replace g's calls; None takes the replace_with of the last bubble_policy().  Returns the corrected CSR ids /
        off / pos_start / pos_end (None without positions) as numpy arrays, or as torch tensors on this handle's device
        written by the device when on_device; and changed (per read: 1 when rewritten) and branch_rewritten (per
        branch: its reads rewritten) as numpy arrays, or with flags_on_device (and on_device) as device tensors of
        uint8 and int32"""
        NB = self.bubble_counts()[1]
        rw = self._replace_with_arg(replace_with, NB, "correct_bubble_reads")
        return self._corrected_csr(lambda *a: self._lib.amira_gmg_correct_bubble_reads(self._h, _ptr(rw), *a),
                                   {"branch_rewritten": NB}, on_device, flags_on_device)

    @staticmethod
    def _replace_with_arg(replace_with, NB, name):
        """replace_with as the C ABI takes it (None stays None), checked for its length and range"""
        if replace_with is None:
            return None
        rw = np.asarray(replace_with, np.int64).ravel()
        if len(rw) != NB or (len(rw) and (rw.min() < -1 or rw.max() >= NB)):
            raise ValueError("%s: replace_with must hold -1 or a branch index for each of %d branches" % (name, NB))
        return np.ascontiguousarray(rw, np.int32)

    @staticmethod
    def _clip_arg(clip, Q, name):
        """clip flags as the C ABI takes them (None stays None), checked for their length and values"""
        if clip is None:
            return None
        cf = np.asarray(clip).ravel()
        if len(cf) != Q or (len(cf) and not np.isin(cf, (0, 1)).all()):
            raise ValueError("%s: clip must hold 0 or 1 for each of %d tips" % (name, Q))
        return np.ascontiguousarray(cf, np.uint8)

    def _corrected_csr(self, call, counts, on_device, flags_on_device) -> dict:
        """the size pass and the fill pass of a correction call (n_calls, read_off, ids, pos_start, pos_end, changed,
        one array per entry of `counts`, out_on_device) -> the dict correct_bubble_reads, clip_tip_reads and
        clean_reads return, with the per item counts under the names of `counts` ({name: number of items})"""
        n = C.c_int64()
        _lib.check(call(C.byref(n), *[None] * (5 + len(counts)), 0))
        G, R = n.value, self.R
        if on_device:
            import torch
            dev = torch.device("cuda", self.device)
            new = lambda size, dt: torch.empty(size, dtype=getattr(torch, dt), device=dev)
        else:
            new = lambda size, dt: np.empty(size, dt)
        a = {"ids": new(G, "int32"), "off": new(R + 1, "int64"),
             "pos_start": new(G, "int32") if self.has_pos else None, "pos_end": new(G, "int32") if self.has_pos else None,
             "changed": np.empty(R, np.uint8), **{f: np.empty(m, np.uint32) for f, m in counts.items()}}
        if on_device:                                                        # per item counts < 2^31, as uint32
            changed, per_item = new(R, "uint8"), {f: new(m, "int32") for f, m in counts.items()}
        else:
            changed, per_item = a["changed"], {f: a[f] for f in counts}
        _lib.check(call(None, _ptr(a["off"]), _ptr(a["ids"]), _ptr(a["pos_start"]), _ptr(a["pos_end"]), _ptr(changed),
                        *[_ptr(per_item[f]) for f in counts], int(bool(on_device))))
        if on_device and flags_on_device:
            a["changed"] = changed
            a.update(per_item)
        elif on_device:
            a["changed"][:] = changed.cpu().numpy()
            for f in counts:
                a[f][:] = per_item[f].cpu().numpy().view(np.uint32)
        return a

    def tips(self) -> dict:
        """the dead-end tips of the compacted graph (amira_gmg_tips), by unitig: per tip its unitig, orientation (+1: a
        walk from the junction into the tip follows the unitig's listed order), attach state (the state of the junction
        node a walk leaves through into the tip) and the read steps on it"""
        Q = C.c_int64()
        _lib.check(self._lib.amira_gmg_tips(self._h, C.byref(Q), *[None] * 4))
        Q = Q.value
        a = {"tip_unitig": np.empty(Q, np.int32), "tip_orient": np.empty(Q, np.int8), "tip_attach": np.empty(Q, np.int32),
             "tip_reads": np.empty(Q, np.uint32)}
        _lib.check(self._lib.amira_gmg_tips(self._h, None, *[_ptr(a[f]) for f in TIP_FIELDS]))
        return a

    def tip_count(self) -> int:
        """the number of tips(), without exporting them"""
        Q = C.c_int64()
        _lib.check(self._lib.amira_gmg_tips(self._h, C.byref(Q), *[None] * 4))
        return Q.value

    def tip_policy(self, min_length: int, ranks=(), want_clip: bool = False):
        """the clipping policy over tips() (amira_gmg_tip_policy): a tip is clipped when it has fewer than min_length
        nodes, no node holding a gene of `ranks` (vocabulary ranks), and a sibling at its junction leads into a unitig of
        strictly larger mean node coverage.  min_length = k + 1 covers single errors in a read's first or last k calls.
        Returns the number of tips clipped, and with want_clip also clip (per tip: 1 or 0) as a numpy array.  The device
        keeps the flags for clip_tip_reads(None)."""
        r = np.ascontiguousarray(ranks, np.int32)
        n = C.c_int64()
        _lib.check(self._lib.amira_gmg_tip_policy(self._h, int(min_length), _ptr(r), len(r), C.byref(n), None))
        if not want_clip:
            return n.value
        clip = np.empty(self.tip_count(), np.uint8)
        if len(clip):
            _lib.check(self._lib.amira_gmg_tip_policy(self._h, int(min_length), _ptr(r), len(r), None, _ptr(clip)))
        return n.value, clip

    def clip_tip_reads(self, clip=None, on_device: bool = False, flags_on_device: bool = False) -> dict:
        """the reads that run into clipped tips, clipped (amira_gmg_clip_tip_reads): clip[q] = 1 clips tip q of tips(),
        0 leaves it; None takes the flags of the last tip_policy().  An end clip drops the calls a read's last step
        holds on the tip, a start clip those of its first step.  Returns the clipped CSR and changed as
        correct_bubble_reads does, with tip_clipped (per tip: the read steps clipped) in place of branch_rewritten"""
        Q = self.tip_count()
        cf = self._clip_arg(clip, Q, "clip_tip_reads")
        return self._corrected_csr(lambda *a: self._lib.amira_gmg_clip_tip_reads(self._h, _ptr(cf), *a),
                                   {"tip_clipped": Q}, on_device, flags_on_device)

    def clean_reads(self, replace_with=None, clip=None, on_device: bool = False, flags_on_device: bool = False) -> dict:
        """the reads cleaned of bubbles and tips in one pass (amira_gmg_clean_reads): the edits of
        correct_bubble_reads(replace_with) and the clips of clip_tip_reads(clip) on this graph, written as one CSR (no
        call is both edited and clipped).  None takes the held replace_with of the last bubble_policy() or the held
        flags of the last tip_policy().  Returns the CSR and changed as correct_bubble_reads does, with both
        branch_rewritten and tip_clipped"""
        NB, Q = self.bubble_counts()[1], self.tip_count()
        rw = self._replace_with_arg(replace_with, NB, "clean_reads")
        cf = self._clip_arg(clip, Q, "clean_reads")
        return self._corrected_csr(lambda *a: self._lib.amira_gmg_clean_reads(self._h, _ptr(rw), _ptr(cf), *a),
                                   {"branch_rewritten": NB, "tip_clipped": Q}, on_device, flags_on_device)

    def gene_paths(self, ranks) -> dict:
        """the reads grouped by their path through the genes of `ranks` (vocabulary ranks; amira_gmg_gene_paths): per
        occurrence (a maximal run of a read's windows on nodes holding one of the genes) its read, first window, length
        in windows, flanks (1 left, 2 right), orientation and cluster (-1 unassigned, -2 ambiguous); per cluster of
        complete occurrences its key key_state[key_off[c]:key_off[c + 1]], its complete occurrences n_complete[c] and
        its members members[member_off[c]:member_off[c + 1]] (occurrence indices, ascending)"""
        r = np.ascontiguousarray(ranks, np.int32)
        n = [C.c_int64() for _ in range(4)]
        _lib.check(self._lib.amira_gmg_gene_paths(self._h, _ptr(r), len(r), *[C.byref(x) for x in n], *[None] * 11))
        O, Cn, KS, M = (x.value for x in n)
        size = {"key_off": Cn + 1, "key_state": KS, "n_complete": Cn, "member_off": Cn + 1, "members": M}
        a = {f: np.zeros(size.get(f, O), t) for f, t in GENE_PATH_FIELDS}
        _lib.check(self._lib.amira_gmg_gene_paths(self._h, _ptr(r), len(r), None, None, None, None,
                                                  *[_ptr(a[f]) for f, _ in GENE_PATH_FIELDS]))
        return a

    def filter_masks(self):
        """keep flags of the last filter / component removal, indexed by the pre-filter node / edge order"""
        a, b = C.c_int64(), C.c_int64()
        _lib.check(self._lib.amira_gmg_filter_mask_sizes(self._h, C.byref(a), C.byref(b)))
        nk, ek = np.ones(a.value, np.int32), np.ones(b.value, np.int32)
        _lib.check(self._lib.amira_gmg_export_filter_masks(self._h, _ptr(nk), _ptr(ek)))
        return nk.astype(bool), ek.astype(bool)

    def sizes(self) -> dict:
        v = [C.c_int64() for _ in range(7)]
        _lib.check(self._lib.amira_gmg_sizes(self._h, *[C.byref(x) for x in v]))
        names = ("nodes", "edges", "windows", "incidences", "fw", "bw", "short_reads")
        return dict(zip(names, (x.value for x in v)))

    def sizes_early(self) -> dict:
        """nodes / edges / windows / short reads: known before the incidence and adjacency passes finish"""
        v = [C.c_int64() for _ in range(4)]
        _lib.check(self._lib.amira_gmg_sizes(self._h, C.byref(v[0]), C.byref(v[1]), C.byref(v[2]), None, None, None,
                                             C.byref(v[3])))
        return dict(zip(("nodes", "edges", "windows", "short_reads"), (x.value for x in v)))

    def phase_ms(self) -> dict:
        out = {}
        for i, name in enumerate(_lib.PHASES):
            ms = C.c_float()
            _lib.check(self._lib.amira_gmg_phase_ms(self._h, i, C.byref(ms)))
            out[name] = ms.value
        return out

    def kernel_launches(self) -> int:
        n = C.c_int64()
        _lib.check(self._lib.amira_gmg_kernel_launches(self._h, C.byref(n)))
        return n.value

    def debug_layout(self, mask: int):
        """test hook: 1 = no 16-byte node slots, 2 = no 16-byte edge slots, 4 = no packed keys, 32 = gene_paths with a
        3-bit key hash (include/amira_gmg.h)"""
        _lib.check(self._lib.amira_gmg_debug_layout(self._h, int(mask)))

    def debug_segsort(self, data, off, out_of_place=False, max_value=None):
        """test hook: sort every segment data[off[s]:off[s+1]] ascending -> (sorted copy, equal neighbours per segment)"""
        data = np.ascontiguousarray(data, np.uint32).copy()
        off = np.ascontiguousarray(off, np.int64)
        dups = np.zeros(len(off) - 1, np.uint32)
        total = C.c_int64()
        _lib.check(self._lib.amira_gmg_debug_segsort(self._h, _ptr(data), _ptr(off), len(off) - 1, _ptr(dups), C.byref(total),
                                                     int(out_of_place), int(data.max()) + 1 if max_value is None and len(data) else int(max_value or 2)))
        return data, dups, total.value

    def atomic_peak(self, table_bytes: int, n_ops: int):
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        _lib.check(self._lib.amira_gmg_atomic_peak(self._h, int(table_bytes), int(n_ops), C.byref(a), C.byref(b),
                                                   C.byref(c)))
        return a.value, b.value, c.value

    # ---- multi-GPU: one process per GPU, contiguous read shards in rank order ----------------------
    def nccl_unique_id(self) -> np.ndarray:
        """128-byte ncclUniqueId (rank 0 creates it, every rank passes it to comm_init)"""
        uid = np.zeros(128, np.uint8)
        _lib.check(self._lib.amira_gmg_nccl_unique_id(_ptr(uid)))
        return uid

    def comm_init(self, unique_id, rank: int, world: int):
        uid = np.ascontiguousarray(unique_id, np.uint8)
        assert uid.size == 128
        _lib.check(self._lib.amira_gmg_comm_init(self._h, _ptr(uid), int(rank), int(world)))
        self.rank, self.world = int(rank), int(world)

    def arrays_reads_only(self) -> dict:
        """only the per-window node indices (what changes in the per-read lists after a removal)"""
        s = self.sizes()
        a = {"win_node": np.empty(s["windows"], np.int32)}
        _lib.check(self._lib.amira_gmg_export_reads(self._h, None, _ptr(a["win_node"]), None, None, None, None, None))
        return a

    def arrays(self, out=None, replicated=True) -> dict:
        """export every graph array to host memory (numpy); `out` may supply preallocated buffers.

        replicated=False (multi-GPU, ranks other than the one that collects the graph): skip the node /
        edge tables every rank holds identically; export only what this rank owns -- its per-read
        lists and its share of the node -> read incidence"""
        early = self.sizes_early()
        n, m, W, R, k = early["nodes"], early["edges"], early["windows"], self.R, self.k

        def buf(name, shape, dtype):
            if out is not None and name in out:
                return out[name]
            return np.empty(shape, dtype)

        a = {
            "k": np.int32(k),
            "win_off": buf("win_off", R + 1, np.int64), "win_node": buf("win_node", W, np.int32),
            "win_dir": buf("win_dir", W, np.int8), "is_short": buf("is_short", R, np.uint8),
            "to_correct": buf("to_correct", R, np.uint8),
        }
        if self.has_pos:
            a["win_start"], a["win_end"] = buf("win_start", W, np.int32), buf("win_end", W, np.int32)
        L = self._lib
        # per-read lists first: they are final before the rest of the build and are copied out beside it
        _lib.check(L.amira_gmg_export_reads(self._h, _ptr(a["win_off"]), _ptr(a["win_node"]), _ptr(a["win_dir"]),
                                            _ptr(a.get("win_start")), _ptr(a.get("win_end")), _ptr(a["is_short"]),
                                            _ptr(a["to_correct"])))
        s = self.sizes()
        if not replicated:
            a.update({"node_reads_off": buf("node_reads_off", n + 1, np.int64),
                      "node_reads": buf("node_reads", s["incidences"], np.int32)})
            _lib.check(L.amira_gmg_export_nodes(self._h, None, None, None, None, _ptr(a["node_reads_off"]),
                                                _ptr(a["node_reads"]), None, None, None, None))
            if n == 0:
                a["node_reads_off"][:] = 0
            return a
        a.update({
            "node_key": buf("node_key", (n, max(k, 0)), np.int32), "node_cov": buf("node_cov", n, np.uint32),
            "node_dir": buf("node_dir", n, np.int8), "node_comp": buf("node_comp", n, np.uint32),
            "node_reads_off": buf("node_reads_off", n + 1, np.int64), "node_reads": buf("node_reads", s["incidences"], np.int32),
            "fw_off": buf("fw_off", n + 1, np.int64), "fw_edges": buf("fw_edges", s["fw"], np.int32),
            "bw_off": buf("bw_off", n + 1, np.int64), "bw_edges": buf("bw_edges", s["bw"], np.int32),
            "edge_src": buf("edge_src", m, np.int32), "edge_tgt": buf("edge_tgt", m, np.int32),
            "edge_sd": buf("edge_sd", m, np.int8), "edge_td": buf("edge_td", m, np.int8), "edge_cov": buf("edge_cov", m, np.uint32),
        })
        _lib.check(L.amira_gmg_export_nodes(self._h, _ptr(a["node_key"]), _ptr(a["node_cov"]), _ptr(a["node_dir"]),
                                            _ptr(a["node_comp"]), _ptr(a["node_reads_off"]), _ptr(a["node_reads"]),
                                            _ptr(a["fw_off"]), _ptr(a["fw_edges"]), _ptr(a["bw_off"]), _ptr(a["bw_edges"])))
        _lib.check(L.amira_gmg_export_edges(self._h, _ptr(a["edge_src"]), _ptr(a["edge_tgt"]), _ptr(a["edge_sd"]),
                                            _ptr(a["edge_td"]), _ptr(a["edge_cov"])))
        if not self.has_pos and out is None:
            a["win_start"] = np.full(W, -1, np.int32)
            a["win_end"] = np.full(W, -1, np.int32)
        if n == 0:
            for f in ("node_reads_off", "fw_off", "bw_off"):
                a[f][:] = 0
        if R == 0:
            a["win_off"][:] = 0
        return a
