"""Gene-call encoding: ``{read_id: ['+geneA', '-geneB', ...]}`` -> signed int32 CSR for the CUDA path.

Replaces, for the whole read set at once, what upstream does one object at a time in
``Gene.__init__`` (amira/construct_gene.py:48-67) and ``convert_genes`` (amira/construct_read.py:5-8).

Gene id = strand * rank, rank in 1..V = position of the gene name in the vocabulary sorted by
``int(sha256(pickle.dumps(name)).hexdigest(), 16)`` ascending.  Upstream orders the genes of a
gene-mer by that integer times the strand (construct_gene.py:91-93, construct_gene_mer.py:15-39);
rank is a monotone map of it, so signed-rank order reproduces the canonical choice exactly.
"""
from __future__ import annotations

import ctypes as C
from itertools import chain

import numpy as np

from . import _lib
from .construct_gene import name_hash


class Vocabulary:
    """gene names in SHA-rank order"""

    def __init__(self, names):
        self.names = sorted(names, key=name_hash)
        self._blob = None

    def __len__(self):
        return len(self.names)

    def blob(self):
        """(utf-8 bytes of all names, int64 byte offsets) for amira_vocab_encode"""
        if self._blob is None:
            enc = [n.encode("utf-8") for n in self.names]
            off = np.zeros(len(enc) + 1, np.int64)
            np.cumsum([len(e) for e in enc], out=off[1:])
            self._blob = (b"".join(enc), off)
        return self._blob

    def sha_bytes(self):
        """(V, 32) uint8: big-endian SHA-256 integer of every gene name, in rank order"""
        if getattr(self, "_sha", None) is None:
            self._sha = np.frombuffer(b"".join(name_hash(n).to_bytes(32, "big") for n in self.names),
                                      np.uint8).reshape(len(self.names), 32)
        return self._sha

    def signed_hashes(self):
        """object array H with H[id + V] = signed SHA int of gene id (index V unused)"""
        V = len(self.names)
        H = np.empty(2 * V + 1, object)
        for r, n in enumerate(self.names, 1):
            h = name_hash(n)
            H[V + r], H[V - r] = h, -h
        return H


def collect_names(reads: dict, toks=None) -> set:
    """unique gene names of a read dict (strand stripped, spaces -> '_'); toks: the flattened calls, if the caller has them"""
    toks = set(chain.from_iterable(reads.values()) if toks is None else toks)
    names = set()
    for t in toks:
        if not isinstance(t, str) or t.replace(" ", "") == "" or t[0] not in "+-" or len(t) < 2:
            continue                      # the encoder reports these with upstream's assertion message
        names.add(t[1:].replace(" ", "_"))
    return names


def encode_reads(reads: dict, vocab: Vocabulary, positions: dict | None = None, toks=None):
    """-> ids int32[G], off int64[R+1], pos_start, pos_end (or None, None)

    Raises AssertionError with upstream's messages for blank tokens, bad strand characters and
    empty names (through the C ABI's status codes), KeyError if a read has no positions entry."""
    lens = np.fromiter(map(len, reads.values()), np.int64, len(reads))
    off = np.zeros(len(reads) + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    G = int(off[-1])
    if toks is None:
        toks = list(chain.from_iterable(reads.values()))
    vblob, voff = vocab.blob()
    ids = np.empty(G, np.int32)
    bad = C.c_int64(-1)
    lib = _lib.load()
    status = None
    try:
        # one blob, newline-separated: the C side splits it (no per-token length pass in Python).  A token with a
        # newline or a NUL in it (no gene name has one) takes the offset form below.
        joined = "\n".join(toks)
    except TypeError:
        _bad_token(next(t for t in toks if not isinstance(t, str)))
    if G and joined.count("\n") == G - 1 and "\0" not in joined:
        status = lib.amira_vocab_encode(joined.encode("utf-8"), None, G, vblob, voff.ctypes.data_as(C.c_void_p), len(vocab),
                                        ids.ctypes.data_as(C.c_void_p), C.byref(bad))
    if status is None:
        blob = "".join(toks).encode("utf-8")
        tok_off = np.zeros(G + 1, np.int64)
        np.cumsum(np.fromiter(map(len, toks), np.int64, G), out=tok_off[1:])
        if len(blob) != int(tok_off[-1]):          # non-ASCII gene names: byte lengths differ from str lengths
            enc = [t.encode("utf-8") for t in toks]
            np.cumsum(np.fromiter(map(len, enc), np.int64, G), out=tok_off[1:])
            blob = b"".join(enc)
        status = lib.amira_vocab_encode(blob, tok_off.ctypes.data_as(C.c_void_p), G, vblob,
                                        voff.ctypes.data_as(C.c_void_p), len(vocab),
                                        ids.ctypes.data_as(C.c_void_p), C.byref(bad))
    _lib.check(status)
    ps = pe = None
    if positions:
        ps = np.empty(G, np.int32)
        pe = np.empty(G, np.int32)
        i = 0
        for rid, calls in reads.items():
            p = positions[rid]
            n = len(calls)
            if n:
                if not p:
                    ps[i:i + n] = -1
                    pe[i:i + n] = -1
                else:
                    arr = np.asarray(p[:n], np.int64).reshape(-1, 2)
                    ps[i:i + n] = arr[:, 0]
                    pe[i:i + n] = arr[:, 1]
            i += n
    return ids, off, ps, pe


def _bad_token(t):
    raise AttributeError("gene calls must be strings, got %r" % (t,))


class EncodedReads:
    """A read set encoded once: vocabulary + signed-id CSR (+ optional positions).

    Amira rebuilds the graph of the same reads many times (k sweep in ``choose_kmer_size``,
    amira/graph_utils.py:258-296; the ~10 rebuilds of ``__main__.py``).  Passing an ``EncodedReads`` to
    ``GeneMerGraph`` in place of the read dict skips the string parsing, and ``device_csr()`` keeps the CSR
    resident on the GPU between builds.  ``save`` / ``load`` are the binary form of upstream's gene-call
    JSON (``process_pandora_json``, amira/pre_processing.py:44-63; ``write_pandora_gene_calls``,
    amira/result_utils.py:1260-1264): an ``.npz`` with the CSR and a vocabulary / read-id sidecar."""

    def __init__(self, reads: dict, positions: dict | None = None):
        self.reads = reads
        self.positions = positions if positions else None
        self.read_ids = list(reads)
        toks = list(chain.from_iterable(reads.values()))
        self.vocab = Vocabulary(collect_names(reads, toks))
        self.ids, self.off, self.pos_start, self.pos_end = encode_reads(reads, self.vocab, self.positions, toks)
        self._device = None

    def __len__(self):
        return len(self.read_ids)

    def device_csr(self, device: int = 0):
        """(ids, off, pos_start, pos_end) as CUDA tensors on `device`, uploaded once"""
        if self._device is None or self._device[0] != device:
            import torch
            dev = torch.device("cuda", device)
            t = lambda a: None if a is None else torch.from_numpy(a).to(dev)
            self._device = (device, t(self.ids), t(self.off), t(self.pos_start), t(self.pos_end))
            torch.cuda.synchronize(dev)
        return self._device[1:]

    def save(self, path: str):
        extra = {} if self.pos_start is None else {"pos_start": self.pos_start, "pos_end": self.pos_end}
        np.savez_compressed(path, ids=self.ids, off=self.off, vocab=np.array(self.vocab.names, dtype=object),
                            read_ids=np.array(self.read_ids, dtype=object), **extra)

    @classmethod
    def load(cls, path: str):
        z = np.load(path, allow_pickle=True)
        self = cls.__new__(cls)
        self.vocab = Vocabulary.__new__(Vocabulary)
        self.vocab.names, self.vocab._blob = [str(n) for n in z["vocab"]], None
        self.read_ids = [str(r) for r in z["read_ids"]]
        self.ids, self.off = z["ids"].astype(np.int32), z["off"].astype(np.int64)
        self.pos_start = z["pos_start"].astype(np.int32) if "pos_start" in z.files else None
        self.pos_end = z["pos_end"].astype(np.int32) if "pos_end" in z.files else None
        self._device = None
        names = self.vocab.names
        toks = [("+" if g > 0 else "-") + names[abs(g) - 1] for g in self.ids.tolist()]
        off = self.off.tolist()
        self.reads = {r: toks[off[i]:off[i + 1]] for i, r in enumerate(self.read_ids)}
        self.positions = None
        if self.pos_start is not None:
            ps, pe = self.pos_start.tolist(), self.pos_end.tolist()
            # encode_reads stores (-1, -1) for the calls of a read whose positions entry is empty: back to []
            self.positions = {r: ([] if off[i + 1] > off[i] and all(ps[j] == -1 and pe[j] == -1 for j in range(off[i], off[i + 1]))
                                  else [(ps[j], pe[j]) for j in range(off[i], off[i + 1])])
                              for i, r in enumerate(self.read_ids)}
        return self

    def corrected(self, out: dict, device: int | None = None):
        """a new EncodedReads over the corrected CSR `out` (GeneMerGraph.correct_compacted_bubbles: ids, off,
        pos_start, pos_end, changed per read, branch_rewritten per branch; GeneMerGraph.clip_compacted_tips: the same
        with tip_clipped per tip in place of branch_rewritten) of these reads.  It shares the vocabulary
        and the read ids; its read / position dicts are shallow copies of these with only the changed reads decoded.
        With torch tensors in `out` (written on GPU `device`) they become its device CSR, and the host CSR is one copy
        of them.  This object is left as it is."""
        new = EncodedReads.__new__(EncodedReads)
        new.vocab, new.read_ids, new._device = self.vocab, self.read_ids, None
        csr = [out[f] for f in ("ids", "off", "pos_start", "pos_end")]
        if not isinstance(csr[0], np.ndarray):
            new._device = (device, *csr)
            csr = [None if x is None else x.cpu().numpy() for x in csr]
        new.ids, new.off, new.pos_start, new.pos_end = csr
        new.changed = np.asarray(out["changed"], np.uint8)
        counts = [f for f in ("branch_rewritten", "tip_clipped") if f in out]
        if not counts:
            raise KeyError("corrected: no branch_rewritten or tip_clipped")
        for f in counts:
            setattr(new, f, np.asarray(out[f], np.uint32))
        new.reads = dict(self.reads)
        new.positions = dict(self.positions) if self.positions is not None else None
        names = self.vocab.names
        for i in np.flatnonzero(new.changed).tolist():
            lo, hi = int(new.off[i]), int(new.off[i + 1])
            rid = self.read_ids[i]
            new.reads[rid] = [("+" if g > 0 else "-") + names[abs(g) - 1] for g in new.ids[lo:hi].tolist()]
            if new.positions is not None and new.positions.get(rid):
                new.positions[rid] = list(zip(new.pos_start[lo:hi].tolist(), new.pos_end[lo:hi].tolist()))
        return new

    def update(self, changed: dict, positions: dict | None = None):
        """Re-encode only the reads in `changed` ({read_id: new gene calls}; the rebuild-after-correction loop of
        iterative_bubble_popping, amira/graph_utils.py:127-181, rewrites a few reads per iteration): the other reads
        keep their encoded calls, the CSR is spliced, and the vocabulary is re-ranked only if a new gene name appears.
        Returns a new EncodedReads over the same (updated in place) read dict."""
        for r in changed:
            if r not in self.reads:
                raise KeyError(r)
        new_names = collect_names(changed) - set(self.vocab.names)
        self.reads.update(changed)
        if positions:
            if self.positions is None:
                self.positions = {}
            self.positions.update(positions)
        if new_names or (positions and self.pos_start is None):
            return EncodedReads(self.reads, self.positions)          # ranks shift: everything is re-encoded
        sub_ids, sub_off, sub_ps, sub_pe = encode_reads(changed, self.vocab, positions if self.pos_start is not None else None)
        index = {r: i for i, r in enumerate(self.read_ids)}
        lens = np.diff(self.off)
        order = [index[r] for r in changed]
        lens[order] = np.diff(sub_off)
        off = np.zeros(len(self.read_ids) + 1, np.int64)
        np.cumsum(lens, out=off[1:])
        out = EncodedReads.__new__(EncodedReads)
        out.reads, out.positions, out.read_ids, out.vocab, out._device = self.reads, self.positions, self.read_ids, self.vocab, None
        out.off = off
        changed_at = dict(zip(order, range(len(order))))

        def splice(old, sub):
            if old is None:
                return None
            new = np.empty(int(off[-1]), old.dtype)
            # unchanged reads in runs between the changed ones
            prev = 0
            for i in sorted(changed_at) + [len(self.read_ids)]:
                if i > prev:
                    new[off[prev]:off[i]] = old[self.off[prev]:self.off[i]]
                if i < len(self.read_ids):
                    j = changed_at[i]
                    new[off[i]:off[i + 1]] = sub[sub_off[j]:sub_off[j + 1]]
                prev = i + 1
            return new
        out.ids = splice(self.ids, sub_ids)
        out.pos_start = splice(self.pos_start, sub_ps if sub_ps is not None else None)
        out.pos_end = splice(self.pos_end, sub_pe if sub_pe is not None else None)
        return out
