"""Seeded synthetic gene-call generator for the BASELINE.json workloads (SURVEY.md section 8d).

Produces the integer CSR form the CUDA path consumes (signed int32 gene ids = strand * SHA-rank,
int64 read offsets) and, for small sizes, the ``{read_id: ['+g', '-h', ...]}`` dict form that the
upstream ``GeneMerGraph`` constructor takes (amira/construct_graph.py:31).

Shape of the data: a gene vocabulary standing in for a panRG; one or more genomes, each a circular
chromosome made of syntenic blocks (a fraction shared between genomes) plus multi-copy plasmids;
a handful of AMR genes inserted at several loci per genome (multi-copy AMR contexts); Zipf genome
abundance; reads are contiguous slices in a random orientation (reverse complement = reversed order,
flipped strands); per-call errors split evenly between false (substituted), missing (deleted) and
strand-flipped calls.

Reads are generated in fixed blocks of ``BLOCK`` reads, each from its own seed, so a rank of a
multi-GPU run can generate exactly its contiguous shard of the global read set.
"""
from __future__ import annotations

import hashlib
import pickle
from dataclasses import dataclass, replace

import numpy as np

BLOCK = 1 << 16


@dataclass(frozen=True)
class SynthConfig:
    name: str
    n_reads: int
    vocab: int
    k: int
    n_genomes: int = 1
    chrom_genes: int = 5400
    n_plasmids: int = 3
    plasmid_genes: int = 200
    shared_frac: float = 0.0       # fraction of 25-gene chromosome blocks shared between genomes
    mean_len: float = 25.0
    fixed_len: int = 0             # >0: every read has exactly this many calls (before deletions)
    max_len: int = 200
    error_rate: float = 0.0
    n_amr: int = 5
    amr_copies: tuple = (2, 6)
    zipf_s: float = 1.1
    seed: int = 0


CONFIGS = {
    # BASELINE.json configs[1..4]
    "c2": SynthConfig("c2_isolate_50k_reads_6k_vocab_k3", 50_000, 6_000, 3, seed=2, error_rate=0.01),
    "c3": SynthConfig("c3_high_error_500k_reads_10pct_k3", 500_000, 6_000, 3, seed=3, error_rate=0.10),
    "c4": SynthConfig("c4_multi_genome_2M_reads_60k_vocab_k3", 2_000_000, 60_000, 3, n_genomes=12,
                      chrom_genes=5000, shared_frac=0.3, seed=4, error_rate=0.01),
    "c5": SynthConfig("c5_metagenome_10M_reads_x30_k5", 10_000_000, 60_000, 5, n_genomes=50,
                      chrom_genes=5000, shared_frac=0.3, fixed_len=30, seed=5, error_rate=0.01),
}


def with_k(cfg: SynthConfig, k: int) -> SynthConfig:
    return replace(cfg, k=k, name=cfg.name.rsplit("_k", 1)[0] + "_k%d" % k)


def vocabulary_names(vocab: int) -> list:
    """synthetic gene names ordered by ascending int(sha256(pickle(name))): rank r -> names[r-1]

    (amira/construct_gene.py:5-10 defines the order that decides which orientation is canonical.)
    """
    names = ["syn%06d" % i for i in range(vocab)]
    for i in range(0, vocab, 997):           # sprinkle AMR-looking names into the vocabulary
        names[i] = "blaSYN-%d" % i
    key = {n: hashlib.sha256(pickle.dumps(n)).digest() for n in names}
    return sorted(names, key=key.get)


class _Pool:
    """all replicons of all genomes, each stored twice back to back so circular slices are contiguous"""

    def __init__(self, cfg: SynthConfig):
        rng = np.random.default_rng([cfg.seed, 0xA111])
        V = cfg.vocab
        blk = 25
        n_blocks = max(1, cfg.chrom_genes // blk)
        backbone = rng.permutation(V)[: n_blocks * blk].astype(np.int32) + 1
        backbone *= rng.choice(np.array([-1, 1], np.int32), size=backbone.size)
        amr = rng.choice(V, size=cfg.n_amr, replace=False).astype(np.int32) + 1
        self.amr = amr                                     # the AMR genes' ranks, and their loci over all genomes
        self.amr_loci = np.zeros(cfg.n_amr, np.int64)
        seqs, genome_of, weight = [], [], []
        for g in range(cfg.n_genomes):
            chrom = backbone.copy().reshape(n_blocks, blk)
            if cfg.n_genomes > 1:
                own = rng.random(n_blocks) >= cfg.shared_frac
                repl = rng.permutation(V)[: int(own.sum()) * blk].astype(np.int32) + 1
                repl *= rng.choice(np.array([-1, 1], np.int32), size=repl.size)
                chrom[own] = repl.reshape(-1, blk)
                order = rng.permutation(n_blocks)          # block rearrangements between genomes
                flip = rng.random(n_blocks) < 0.2
                chrom = [(-c[::-1] if f else c) for c, f in zip(chrom[order], flip[order])]
                chrom = np.concatenate(chrom)
            else:
                chrom = chrom.reshape(-1)
            reps = [chrom]
            for _ in range(cfg.n_plasmids):
                p = rng.permutation(V)[: cfg.plasmid_genes].astype(np.int32) + 1
                p *= rng.choice(np.array([-1, 1], np.int32), size=p.size)
                reps.append(p)
            # multi-copy AMR contexts: each AMR gene dropped into several loci of this genome
            for ai, a in enumerate(amr):
                n_copy = int(rng.integers(cfg.amr_copies[0], cfg.amr_copies[1] + 1))
                self.amr_loci[ai] += n_copy
                for _ in range(n_copy):
                    ri = int(rng.integers(0, len(reps)))
                    at = int(rng.integers(0, len(reps[ri]) + 1))
                    reps[ri] = np.insert(reps[ri], at, a * int(rng.choice([-1, 1])))
            for ri, s in enumerate(reps):
                copies = 1.0 if ri == 0 else float(rng.integers(1, 6))
                seqs.append(s.astype(np.int32))
                genome_of.append(g)
                weight.append(len(s) * copies)
        self.lens = np.array([len(s) for s in seqs], np.int64)
        self.base = np.concatenate([[0], np.cumsum(2 * self.lens)])[:-1]
        self.pool = np.concatenate([np.concatenate([s, s]) for s in seqs])
        abundance = 1.0 / np.arange(1, cfg.n_genomes + 1) ** cfg.zipf_s
        w = np.array(weight) * abundance[np.array(genome_of)]
        self.cdf = np.cumsum(w / w.sum())


_POOLS = {}


def _pool(cfg: SynthConfig) -> _Pool:
    key = replace(cfg, n_reads=0, k=0, name="", error_rate=0.0)
    if key not in _POOLS:
        _POOLS.clear()
        _POOLS[key] = _Pool(cfg)
    return _POOLS[key]


def _block(cfg: SynthConfig, pool: _Pool, b: int, n: int):
    rng = np.random.default_rng([cfg.seed, 0xB10C, b])
    rep = np.minimum(np.searchsorted(pool.cdf, rng.random(n)), len(pool.lens) - 1)
    rlen = pool.lens[rep]
    if cfg.fixed_len:
        L = np.full(n, cfg.fixed_len, np.int64)
    else:
        sigma = 0.6
        L = np.rint(rng.lognormal(np.log(cfg.mean_len) - sigma * sigma / 2, sigma, n)).astype(np.int64)
        L = np.clip(L, 1, cfg.max_len)
    L = np.minimum(L, rlen)
    start = (rng.random(n) * rlen).astype(np.int64)
    rev = rng.random(n) < 0.5
    off = np.zeros(n + 1, np.int64)
    np.cumsum(L, out=off[1:])
    G = int(off[-1])
    j = np.arange(G, dtype=np.int64) - np.repeat(off[:-1], L)
    revg = np.repeat(rev, L)
    j = np.where(revg, np.repeat(L, L) - 1 - j, j)
    ids = pool.pool[np.repeat(pool.base[rep] + start, L) + j]
    ids = np.where(revg, -ids, ids).astype(np.int32)
    if cfg.error_rate > 0:
        u = rng.random(G)
        bad = u < cfg.error_rate
        kind = rng.integers(0, 3, G)
        sub = bad & (kind == 0)
        ids[sub] = (rng.integers(1, cfg.vocab + 1, int(sub.sum())) *
                    rng.choice(np.array([-1, 1]), int(sub.sum()))).astype(np.int32)
        flip = bad & (kind == 2)
        ids[flip] = -ids[flip]
        keep = ~(bad & (kind == 1))
        kept = np.concatenate([[0], np.cumsum(keep)])
        off = kept[off]
        ids = ids[keep]
    return ids, off


def generate(cfg: SynthConfig, first_read: int = 0, n_reads: int | None = None):
    """(ids int32[G], off int64[R+1]) for reads [first_read, first_read + n_reads) of the config"""
    if n_reads is None:
        n_reads = cfg.n_reads - first_read
    pool = _pool(cfg)
    ids_parts, off_parts, total = [], [np.zeros(1, np.int64)], 0
    r = first_read
    end = first_read + n_reads
    while r < end:
        b = r // BLOCK
        lo, hi = b * BLOCK, min((b + 1) * BLOCK, cfg.n_reads)
        ids, off = _block(cfg, pool, b, hi - lo)
        a, z = r - lo, min(end, hi) - lo
        ids_parts.append(ids[off[a]:off[z]])
        off_parts.append(off[a + 1:z + 1] - off[a] + total)
        total += int(off[z] - off[a])
        r = lo + z
    ids = np.concatenate(ids_parts) if ids_parts else np.zeros(0, np.int32)
    return np.ascontiguousarray(ids, np.int32), np.concatenate(off_parts).astype(np.int64)


def count_windows(off: np.ndarray, k: int) -> int:
    L = np.diff(off)
    return int(np.maximum(L - (k - 1), 0).sum())


def to_read_dict(ids: np.ndarray, off: np.ndarray, names: list, first_read: int = 0) -> dict:
    """integer CSR -> the dict-of-strings the upstream constructor takes (small inputs only)"""
    toks = [("+" if x > 0 else "-") + names[abs(int(x)) - 1] for x in ids.tolist()]
    return {"read%09d" % (first_read + i): toks[off[i]:off[i + 1]] for i in range(len(off) - 1)}


def positions_for(off: np.ndarray, seed: int = 0):
    """plausible per-call (start, end) read coordinates: ~1 kb genes with small gaps"""
    rng = np.random.default_rng([seed, 0x9051])
    G = int(off[-1])
    glen = rng.integers(300, 1500, G)
    gap = rng.integers(0, 200, G)
    step = glen + gap
    c = np.cumsum(step) - step
    first = np.repeat(c[off[:-1].clip(max=max(G - 1, 0))] if G else np.zeros(0, np.int64), np.diff(off))
    start = (c - first + gap).astype(np.int32)
    return start, (start + glen).astype(np.int32)
