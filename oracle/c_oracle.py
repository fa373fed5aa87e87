"""ctypes binding of the plain-C oracle (oracle/gmg_oracle.c) -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs use it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libgmg_oracle.so")
_lib = None

E_PALINDROME, E_NOMEM, E_MULTIEDGE, E_BADARG = 1, 2, 3, 4


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "gmg_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-shared", "-o", _SO, src])
    return _SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        _lib = C.CDLL(_SO)
        _lib.oracle_build.restype = C.c_int
        _lib.oracle_filter.restype = C.c_int
        _lib.oracle_remove_low_coverage_components.restype = C.c_int
        _lib.oracle_remove_nodes.restype = C.c_int
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class COracleGraph:
    def __init__(self, ids, off, k, pos_start=None, pos_end=None):
        self.ids = np.ascontiguousarray(ids, np.int32)
        self.off = np.ascontiguousarray(off, np.int64)
        self.k = int(k)
        self.R = len(self.off) - 1
        self.has_pos = pos_start is not None
        ps = None if pos_start is None else np.ascontiguousarray(pos_start, np.int32)
        pe = None if pos_end is None else np.ascontiguousarray(pos_end, np.int32)
        self._h = C.c_void_p()
        rc = lib().oracle_build(C.byref(self._h), _p(self.ids), _p(self.off), C.c_int64(self.R),
                                C.c_int32(self.k), _p(ps), _p(pe))
        if rc == E_PALINDROME:
            raise AssertionError("Gene-mer and reverse complement gene-mer are identical")
        if rc == E_BADARG:
            raise AssertionError("Gene-mer is empty")
        if rc:
            raise MemoryError("oracle_build failed: %d" % rc)

    def filter_graph(self, min_node_cov, min_edge_cov):
        lib().oracle_filter(self._h, C.c_uint32(min_node_cov), C.c_uint32(min_edge_cov))
        return self

    def remove_low_coverage_components(self, c):
        rc = lib().oracle_remove_low_coverage_components(self._h, C.c_uint32(c))
        if rc == E_MULTIEDGE:
            raise TypeError("unhashable type: 'list'")

    def remove_nodes(self, flags):
        """remove_node for every node whose flag is set (flags[n_nodes], current node order); TypeError and no
        change when one of them has two edges to the same neighbour"""
        f = np.ascontiguousarray(flags, np.uint8)
        n = C.c_int64()
        lib().oracle_sizes(self._h, C.byref(n), *[C.byref(C.c_int64()) for _ in range(5)])
        assert f.shape == (n.value,), (f.shape, n.value)
        if lib().oracle_remove_nodes(self._h, _p(f)) == E_MULTIEDGE:
            raise TypeError("unhashable type: 'list'")

    def arrays(self) -> dict:
        L = lib()
        s = [C.c_int64() for _ in range(6)]
        L.oracle_sizes(self._h, *[C.byref(x) for x in s])
        n, m, W, ninc, nfw, nbw = [x.value for x in s]
        k = self.k
        a = {
            "k": np.int32(k),
            "node_key": np.zeros((n, max(k, 0)), np.int32), "node_cov": np.zeros(n, np.uint32),
            "node_dir": np.zeros(n, np.int8), "node_comp": np.zeros(n, np.uint32),
            "node_reads_off": np.zeros(n + 1, np.int64), "node_reads": np.zeros(ninc, np.int32),
            "fw_off": np.zeros(n + 1, np.int64), "fw_edges": np.zeros(nfw, np.int32),
            "bw_off": np.zeros(n + 1, np.int64), "bw_edges": np.zeros(nbw, np.int32),
            "edge_src": np.zeros(m, np.int32), "edge_tgt": np.zeros(m, np.int32),
            "edge_sd": np.zeros(m, np.int8), "edge_td": np.zeros(m, np.int8), "edge_cov": np.zeros(m, np.uint32),
            "win_off": np.zeros(self.R + 1, np.int64), "win_node": np.zeros(W, np.int32),
            "win_dir": np.zeros(W, np.int8), "win_start": np.zeros(W, np.int32), "win_end": np.zeros(W, np.int32),
            "is_short": np.zeros(self.R, np.uint8), "to_correct": np.zeros(self.R, np.uint8),
        }
        L.oracle_export_nodes(self._h, _p(a["node_key"]), _p(a["node_cov"]), _p(a["node_dir"]), _p(a["node_comp"]),
                              _p(a["node_reads_off"]), _p(a["node_reads"]), _p(a["fw_off"]), _p(a["fw_edges"]),
                              _p(a["bw_off"]), _p(a["bw_edges"]))
        L.oracle_export_edges(self._h, _p(a["edge_src"]), _p(a["edge_tgt"]), _p(a["edge_sd"]), _p(a["edge_td"]),
                              _p(a["edge_cov"]))
        L.oracle_export_reads(self._h, _p(a["win_off"]), _p(a["win_node"]), _p(a["win_dir"]), _p(a["win_start"]),
                              _p(a["win_end"]), _p(a["is_short"]), _p(a["to_correct"]))
        return a

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.oracle_free(self._h)
            self._h = None
