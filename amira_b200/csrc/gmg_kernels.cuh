// gmg_kernels.cuh -- hand-written sm_100a kernels of the GeneMerGraph build.
//
// Upstream (pure Python) walks reads one at a time and does ~28 SHA-256 per gene-mer
// (amira/construct_graph.py:45-100).  Here the reads are a CSR of signed int32 gene ids and the
// whole build is a handful of data-parallel passes:
//
//   k_read_windows     per read: window count (construct_read.py:41-43), short-read flag, and the
//                      read that owns each 128-call chunk boundary
//   k_insert_windows   THE hot kernel (this file).  One warp per 128-call chunk, no block barriers:
//                      128-bit staging of the chunk (+k halo) in per-warp shared memory, read
//                      boundaries by a warp max-scan, per-window canonicalisation against the reverse
//                      complement (construct_gene_mer.py:4-39), hash, insert into the node table with
//                      first-seen tracking (atomicCAS / atomicMin on one 64-bit word), coverage
//                      RED.ADD, per-window outputs, then adjacent-pair edges from the slot numbers
//                      staged in shared memory (construct_graph.py:246-324), two probes in flight per lane
//   post_kernels.cuh   first-seen order without a sort (a bitmap over call positions + a prefix popcount
//                      gives every node / edge its rank in upstream's dict order), node / edge arrays
//                      written coalesced through an inverse map, adjacency, connected components over
//                      runs of consecutive nodes with a lock-free union-find (construct_graph.py:911-927),
//                      filters: thresholds + order-preserving stream compaction (:496-540, 950-958)
//   incidence.cuh      per-read node lists (construct_graph.py:165-178) and node -> unique ascending reads
//                      (construct_node.py:64-67): a partition pass into per-unit buckets + one CTA per
//                      unit sorting its lists in shared memory
//   segsort.cuh        segmented sorts (adjacency lists; read lists beyond one CTA's shared memory)
//   scan.cuh           single-pass look-back scans with device-side element counts
//   stats.cuh          the post-build scans of the callers
//   unitigs.cuh        the compacted graph by list ranking; its junction edges as links between unitig ends, and
//                      the reads as steps along unitigs (one scan over the windows)
//   bubbles.cuh        the simple bubbles of the compacted graph (branches per edge, grouping per list by warp),
//                      and the popping policy (one warp per bubble)
//   correct.cuh        the reads through the bubbles rewritten along a kept branch (edits per step, one scan
//                      over the calls)
//   sharded.cuh        the multi-GPU exchange and merge
#pragma once

#include "common.cuh"
#include "scan.cuh"
#include "segsort.cuh"

namespace amira {

constexpr int INS_THREADS = 256;
constexpr int INS_WARPS = INS_THREADS / 32;
constexpr int WC = 128;        // calls per warp chunk
constexpr int INS_TILE = WC;   // granularity of the chunk -> first read map
constexpr int MAX_K = 64;
#ifndef AMIRA_INS_MINB
#define AMIRA_INS_MINB 6
#endif
constexpr int NR_STAGE = 30;   // reads of a chunk whose offsets are staged in shared memory
constexpr unsigned int INVALID_VAL = 0xFFFFFFFFu;
constexpr unsigned int MAX_PROBES = 1u << 15;

// device-side status words; ST_STALE: the call count assumed by the host (cached from an earlier build of
// the same device-resident offsets) no longer matches read_off[R]; ST_MAXABS: largest |gene id| staged
enum { ST_ERR = 0, ST_OVERFLOW_N = 1, ST_OVERFLOW_E = 2, ST_UNPACK = 3, ST_STALE = 4, ST_MAXABS = 5, ST_COUNT = 8 };
// device-side sizes (the host reads them once, when the caller first asks for a size or an export)
enum { SZ_W = 0, SZ_NODES = 1, SZ_EDGES = 2, SZ_INC = 3, SZ_SHORT = 4, SZ_FW = 5, SZ_BW = 6, SZ_DUPS = 7,
       SZ_COMPS = 8, SZ_COUNT = 16 };

struct BuildParams {
    const int32_t *ids;
    const int64_t *off;
    const int64_t *win_off;
    const int32_t *tile_r0;
    const int32_t *ps;
    const int32_t *pe;
    int64_t G, R, n_tiles;
    int64_t tile_lo, tile_hi;  // chunks this launch covers (the host streams the ids in and launches per piece)
    int k;
    NodeSlot *ntab;      // 32-byte node slots (or NodeSlot16 *ntab16 + ncov when the gene-mers fit 85 bits)
    NodeSlot16 *ntab16;
    unsigned int *ncov;  // coverage side array of the 16-byte layout (counts from 0xFFFFFFFF)
    unsigned int ncap;
    EdgeSlot *etab;      // 32-byte edge slots (or EdgeSlot16 *etab16 when call positions fit 30 bits)
    EdgeSlot16 *etab16;
    unsigned int ecap;
    int32_t *win_node;
    int8_t *win_dir;
    int32_t *win_read;   // read of the window (global index)
    int32_t *win_start;
    int32_t *win_end;
    int *status;
    int64_t read_base;  // global index of this shard's first read (multi-GPU)
    int key_bits;       // bits per gene of the packed key (<= 124 bits); 0: gene-mers are compared through ids
    int ids_aligned;    // ids is 16-byte aligned (128-bit staging loads)
};

__host__ __device__ __forceinline__ int64_t imin64(int64_t a, int64_t b) { return a < b ? a : b; }

struct MaxOp {
    __device__ __forceinline__ int operator()(int a, int b) const { return a > b ? a : b; }
};

// ---------------------------------------------------------------------------------------------
__global__ void k_read_windows(const int64_t *__restrict__ off, int64_t R, int k, int64_t G,
                               int64_t *__restrict__ nwin, uint8_t *__restrict__ is_short,
                               uint8_t *__restrict__ to_correct, int32_t *__restrict__ tile_r0,
                               long long *__restrict__ sizes, int *__restrict__ status) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool shortr = false;
    if (r < R) {
        int64_t a = off[r], b = off[r + 1];
        if (b < a || a < 0 || b > G) {
            status[ST_ERR] = AMIRA_E_ARG;
            b = a;
        }
        int64_t L = b - a;
        int64_t nw = L >= k ? L - k + 1 : 0;
        nwin[r] = nw;
        shortr = nw == 0;
        is_short[r] = shortr;
        to_correct[r] = 0;
        // this read owns every tile whose first call lies inside it
        for (int64_t t = (a + INS_TILE - 1) / INS_TILE; t * INS_TILE < b; ++t) tile_r0[t] = (int32_t)r;
    } else if (r == R) {
        nwin[R] = 0;
        if (R > 0 && off[R] != G) status[ST_STALE] = 1;  // the host's (cached) call count is out of date
    }
    unsigned m = __ballot_sync(0xffffffffu, shortr);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd((unsigned long long *)&sizes[SZ_SHORT], (unsigned long long)__popc(m));
}

// ---------------------------------------------------------------------------------------------
// hash of the canonical form of a window (dirneg: the window is the reverse complement of it)
__device__ __forceinline__ unsigned long long canonical_hash(const int32_t *win, int k, int dirneg) {
    unsigned long long h = 0x9e3779b97f4a7c15ULL;
    for (int i = 0; i < k; ++i) {
        int g = dirneg ? -win[k - 1 - i] : win[i];
        h = (h ^ (unsigned long long)(unsigned int)g) * 0x100000001b3ULL;
        h ^= h >> 29;
    }
    return mix64(h);
}

__device__ __forceinline__ unsigned long long packed_hash(unsigned long long klo, unsigned long long khi) {
    unsigned long long h = (klo * 0x9E3779B97F4A7C15ULL) ^ ((khi + 0x632BE59BD9B4E019ULL) * 0xC2B2AE3D27D4EB4FULL);
    h ^= h >> 32;
    h *= 0xD6E8FEB86659FD93ULL;
    h ^= h >> 29;
    return h;
}

// 32-bit bucket hash of a packed key of at most 85 bits (the 16-byte layout: the key itself is the identity, the
// hash only picks the bucket): 32-bit multiplies instead of the three 64-bit ones of packed_hash
__device__ __forceinline__ unsigned int packed_hash32(unsigned long long klo, unsigned long long khi) {
    unsigned int h = (unsigned int)klo * 0x9E3779B1u;
    h ^= h >> 15;
    h += (unsigned int)(klo >> 32) * 0x85EBCA77u;
    h ^= h >> 13;
    h += (unsigned int)khi * 0xC2B2AE3Du;
    h *= 0x27D4EB2Fu;
    h ^= h >> 16;
    h *= 0x165667B1u;
    h ^= h >> 15;
    return h;
}

__device__ __forceinline__ unsigned int edge_hash32(unsigned long long key) {
    unsigned int h = (unsigned int)key * 0x9E3779B1u;
    h ^= h >> 15;
    h += (unsigned int)(key >> 32) * 0x85EBCA77u;
    h ^= h >> 13;
    h *= 0x27D4EB2Fu;
    h ^= h >> 16;
    h *= 0x165667B1u;
    h ^= h >> 15;
    return h;
}

// one 256-bit load of a node slot (LDG.E.256): word, cov|aux, packed key halves
__device__ __forceinline__ void load_node_slot(const NodeSlot *s, unsigned long long &word, unsigned long long &ca,
                                               unsigned long long &klo, unsigned long long &khi) {
    asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(word), "=l"(ca), "=l"(klo), "=l"(khi) : "l"(s));
}

__device__ __forceinline__ void publish_key(NodeSlot *s, unsigned long long klo, unsigned long long khi) {
    asm volatile("st.global.cg.v2.u64 [%0], {%1,%2};" ::"l"(&s->klo), "l"(klo), "l"(khi) : "memory");
}

__device__ __forceinline__ void load_edge_slot(const EdgeSlot *s, unsigned long long &key, unsigned long long &ord) {
    asm volatile("ld.global.cg.v2.u64 {%0,%1}, [%2];" : "=l"(key), "=l"(ord) : "l"(s));
}

// compare a window (canonical form given by win / dirneg) with the representative window of a slot
__device__ __forceinline__ bool same_as_representative(const BuildParams &P, const int32_t *win, int dirneg,
                                                       unsigned long long cur) {
    const int k = P.k;
    const int64_t q = (int64_t)((cur >> 1) & P_MASK);
    const int qneg = (int)(cur & 1ull);
    for (int j = 0; j < k; ++j) {
        int a = dirneg ? -win[k - 1 - j] : win[j];
        int b = qneg ? -__ldg(P.ids + q + (k - 1 - j)) : __ldg(P.ids + q + j);
        if (a != b) return false;
    }
    return true;
}

// Node table insert-or-find.  The slot is claimed by a CAS on `word` (fingerprint | first call
// position | first direction); the winner then publishes the packed key (<= 124 bits) in the same 32-byte
// sector, so that every later visitor decides "same gene-mer?" from the one sector it loaded.
// Until the key is published (or when the gene-mer does not fit 124 bits: packed == false) the
// comparison falls back to the representative window ids[p .. p+k) named by `word`.
__device__ __forceinline__ unsigned int node_insert(const BuildParams &P, const int32_t *win, int dirneg, bool packed,
                                                    unsigned long long klo, unsigned long long khi,
                                                    unsigned long long h, unsigned long long mine) {
    const unsigned int cap = P.ncap;
    unsigned int s = (unsigned int)(((unsigned long long)(unsigned int)h * cap) >> 32);
    const unsigned int fp = (unsigned int)(mine >> FP_SHIFT);
    const unsigned int max_probe = min(MAX_PROBES, cap);
    for (unsigned int probe = 0; probe < max_probe; ++probe) {
        unsigned long long cur, ca, sl, sh;
        load_node_slot(&P.ntab[s], cur, ca, sl, sh);
        if (cur == EMPTY64) {
            unsigned long long old = atomicCAS(&P.ntab[s].word, EMPTY64, mine);
            if (old == EMPTY64) {
                if (packed) publish_key(&P.ntab[s], klo, khi);
                return s;
            }
            cur = old;
            sl = sh = EMPTY64;
        }
        bool same;
        if (packed && sl != EMPTY64 && sh != EMPTY64) same = (sl == klo) & (sh == khi);
        else same = ((unsigned int)(cur >> FP_SHIFT) == fp) && same_as_representative(P, win, dirneg, cur);
        if (same) {
            if (mine < cur) atomicMin(&P.ntab[s].word, mine);  // keep the first occurrence
            return s;
        }
        if (++s == cap) s = 0;
    }
    P.status[ST_OVERFLOW_N] = 1;
    return 0;
}

__device__ __forceinline__ void edge_insert(const BuildParams &P, unsigned long long key, unsigned long long ord) {
    const unsigned int cap = P.ecap;
    unsigned long long h = key * 0x9E3779B97F4A7C15ULL;
    h ^= h >> 32;
    h *= 0xD6E8FEB86659FD93ULL;
    unsigned int s = (unsigned int)(h >> 32);
    s = (unsigned int)(((unsigned long long)s * cap) >> 32);
    const unsigned int max_probe = min(MAX_PROBES, cap);
    for (unsigned int probe = 0; probe < max_probe; ++probe) {
        unsigned long long cur, cord;
        load_edge_slot(&P.etab[s], cur, cord);
        if (cur == EMPTY64) {
            unsigned long long old = atomicCAS(&P.etab[s].key, EMPTY64, key);
            cur = (old == EMPTY64) ? key : old;
            cord = EMPTY64;
        }
        if (cur == key) {
            if (ord < cord) atomicMin(&P.etab[s].ord, ord);
            atomicAdd(&P.etab[s].cov, 1u);
            return;
        }
        if (++s == cap) s = 0;
    }
    P.status[ST_OVERFLOW_E] = 1;
}

// ---- 16-byte layouts (see common.cuh) -------------------------------------------------------------
__device__ __forceinline__ void load_slot16(const void *s, unsigned long long &a, unsigned long long &b) {
    asm volatile("ld.global.cg.v2.u64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(s));
}

__device__ __forceinline__ void load_bucket(const void *s, unsigned long long &a0, unsigned long long &b0,
                                            unsigned long long &a1, unsigned long long &b1) {
    asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(a0), "=l"(b0), "=l"(a1), "=l"(b1) : "l"(s));
}

// The 16-byte tables are probed by BUCKETS of two slots = one 32-byte sector: one LDG.256 brings
// both, a gene-mer lives in the first free slot of the first bucket with room (slots never empty
// again, so a search stops at the first empty slot).  At 50% load that is ~1.1 sector loads per
// lookup with a short tail, against ~1.5 and a long tail for slot-wise linear probing -- and the
// tail is what a warp pays for, since its lanes wait for the longest probe sequence among them.
//
// mine = (top 22 key bits) << 42 | first position << 1 | first direction; keylow = low 63 key bits
__device__ __forceinline__ unsigned int node_insert16(const BuildParams &P, const int32_t *win, int dirneg,
                                                      unsigned long long keylow, unsigned long long h,
                                                      unsigned long long mine) {
    const unsigned int nb = P.ncap >> 1;
    unsigned int b = (unsigned int)(((unsigned long long)(unsigned int)h * nb) >> 32);
    const unsigned int top = (unsigned int)(mine >> FP_SHIFT);
    const unsigned int max_probe = min(MAX_PROBES, nb);  // a full table is reported after one lap
    for (unsigned int probe = 0; probe < max_probe; ++probe) {
        NodeSlot16 *B = P.ntab16 + 2 * (size_t)b;
        unsigned long long w0, k0, w1, k1;
        load_bucket(B, w0, k0, w1, k1);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            unsigned long long cur = i ? w1 : w0, key = i ? k1 : k0;
            if (cur == EMPTY64) {
                unsigned long long old = atomicCAS(&B[i].word, EMPTY64, mine);
                if (old == EMPTY64) {
                    __stcg(&B[i].key, keylow);
                    return 2 * b + i;
                }
                cur = old;
                key = EMPTY64;
            }
            if ((unsigned int)(cur >> FP_SHIFT) == top) {
                const bool same = (key != EMPTY64) ? (key == keylow) : same_as_representative(P, win, dirneg, cur);
                if (same) {
                    if (mine < cur) atomicMin(&B[i].word, mine);  // keep the first occurrence
                    return 2 * b + i;
                }
            }
        }
        if (++b == nb) b = 0;
    }
    P.status[ST_OVERFLOW_N] = 1;
    return 0;
}

// one bucket of the edge table against `key`: true when the pair event has been counted (found or claimed)
__device__ __forceinline__ bool edge_bucket16(EdgeSlot16 *B, unsigned long long key, unsigned int ord, unsigned long long c0,
                                              unsigned long long o0, unsigned long long c1, unsigned long long o1) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        unsigned long long cur = i ? c1 : c0;
        unsigned int cord = (unsigned int)((i ? o1 : o0) >> 32);
        if (cur == EMPTY64) {
            unsigned long long old = atomicCAS(&B[i].key, EMPTY64, key);
            cur = (old == EMPTY64) ? key : old;
            cord = 0xFFFFFFFFu;
        }
        if (cur == key) {
            if (ord < cord) atomicMin(&B[i].ord, ord);
            atomicAdd(&B[i].cov, 1u);
            return true;
        }
    }
    return false;
}

__device__ __forceinline__ unsigned int edge_bucket_of(const BuildParams &P, unsigned long long key) {
    return (unsigned int)(((unsigned long long)edge_hash32(key) * (P.ecap >> 1)) >> 32);
}

// probe sequence from bucket b on (b itself included)
__device__ __forceinline__ void edge_insert16_from(const BuildParams &P, unsigned long long key, unsigned int ord, unsigned int b) {
    const unsigned int nb = P.ecap >> 1;
    const unsigned int max_probe = min(MAX_PROBES, nb);
    for (unsigned int probe = 0; probe < max_probe; ++probe) {
        if (b >= nb) b = 0;
        EdgeSlot16 *B = P.etab16 + 2 * (size_t)b;
        unsigned long long c0, o0, c1, o1;
        load_bucket(B, c0, o0, c1, o1);
        if (edge_bucket16(B, key, ord, c0, o0, c1, o1)) return;
        ++b;
    }
    P.status[ST_OVERFLOW_E] = 1;
}

__device__ __forceinline__ void edge_insert16(const BuildParams &P, unsigned long long key, unsigned int ord) {
    const unsigned int nb = P.ecap >> 1;
    unsigned int b = (unsigned int)(((unsigned long long)edge_hash32(key) * nb) >> 32);
    const unsigned int max_probe = min(MAX_PROBES, nb);
    for (unsigned int probe = 0; probe < max_probe; ++probe) {
        EdgeSlot16 *B = P.etab16 + 2 * (size_t)b;
        unsigned long long c0, o0, c1, o1;
        load_bucket(B, c0, o0, c1, o1);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            unsigned long long cur = i ? c1 : c0;
            unsigned int cord = (unsigned int)((i ? o1 : o0) >> 32);
            if (cur == EMPTY64) {
                unsigned long long old = atomicCAS(&B[i].key, EMPTY64, key);
                cur = (old == EMPTY64) ? key : old;
                cord = 0xFFFFFFFFu;
            }
            if (cur == key) {
                if (ord < cord) atomicMin(&B[i].ord, ord);
                atomicAdd(&B[i].cov, 1u);
                return;
            }
        }
        if (++b == nb) b = 0;
    }
    P.status[ST_OVERFLOW_E] = 1;
}

// per-warp staging area: one 128-call chunk (+ halo) and what the lanes exchange about it
struct __align__(16) WarpStage {
    int32_t ids[WC + MAX_K + 4];
    int j[WC];                 // read (relative to the chunk's first read) of each call
    unsigned int val[WC + 4];  // slot | dirneg << 31 per window start, INVALID_VAL if none
    long long off[NR_STAGE + 2];
    long long woff[NR_STAGE + 1];
};

// THE hot kernel.  One warp per 128-call chunk, no block-level barriers: every warp stages its chunk
// (+k halo) with 128-bit loads, finds the read of every call with a warp max-scan over the read
// starts that fall in the chunk, canonicalises / packs / hashes each window, inserts into the node
// table, writes the per-window outputs, and inserts the adjacent-pair edges from the slot numbers
// it staged in shared memory.  K > 0: gene-mer size known at compile time (windows in registers).
// N16 / E16: 16-byte node / edge slots.
template <int K, bool N16, bool E16>
__global__ void __launch_bounds__(INS_THREADS, AMIRA_INS_MINB) k_insert_windows(const BuildParams P) {
    __shared__ WarpStage s_stage[INS_WARPS];
    const int lane = threadIdx.x & 31;
    WarpStage &S = s_stage[threadIdx.x >> 5];
    const int k = K ? K : P.k;
    const int kb = P.key_bits;  // bits per gene of the packed key (from the largest |id|), 0 = unpacked
    const bool packed = kb > 0;
    const int64_t n_warps = (int64_t)gridDim.x * INS_WARPS;
    for (int64_t c = P.tile_lo + (int64_t)blockIdx.x * INS_WARPS + (threadIdx.x >> 5); c < P.tile_hi; c += n_warps) {
        const int64_t c0 = c * WC;
        const int len = (int)imin64(WC, P.G - c0);
        const int n_load = (int)imin64(len + k, P.G - c0);
        const int r_lo = P.tile_r0[c];
        const int r_hi = (c + 1 < P.n_tiles) ? P.tile_r0[c + 1] : (int)(P.R - 1);
        const int nr = r_hi - r_lo + 1;

        // ---- stage the chunk (+ halo); c0 is a multiple of 128 calls
        {
            const int32_t *src = P.ids + c0;
            // a packed field holds g + 2^(kb-1); the canonical form also packs -g, and the all-ones and all-zero
            // field values stay free (an all-ones key half means "not published"): |g| <= 2^(kb-1) - 2
            const unsigned int lim = packed ? ((1u << (kb - 1)) - 2u) : 0x7FFFFFFFu;
            unsigned int mx = 0;
            const int i4 = lane * 4;
            if (P.ids_aligned && i4 + 4 <= n_load) {
                const int4 v = __ldcs(reinterpret_cast<const int4 *>(src) + lane);  // streamed once: evict first
                *reinterpret_cast<int4 *>(&S.ids[i4]) = v;
                mx = max(max((unsigned int)abs(v.x), (unsigned int)abs(v.y)), max((unsigned int)abs(v.z), (unsigned int)abs(v.w)));
            } else {
                for (int i = i4; i < i4 + 4 && i < n_load; ++i) {
                    const int g = __ldcs(src + i);
                    S.ids[i] = g;
                    mx = max(mx, (unsigned int)abs(g));
                }
            }
            for (int i = WC + lane; i < n_load; i += 32) {
                const int g = __ldcs(src + i);
                S.ids[i] = g;
                mx = max(mx, (unsigned int)abs(g));
            }
            // abs(INT_MIN) stays 0x80000000 as unsigned: larger than any limit, as it must be
            if (__any_sync(0xffffffffu, mx > lim) && packed) {
                if (mx > lim) P.status[ST_UNPACK] = 1;  // the host redoes the build with wider fields
            }
            // largest |id| of this input, for the key width of the next build on the handle
            mx = __reduce_max_sync(0xffffffffu, mx);
            if (lane == 0 && mx > ((volatile unsigned int *)P.status)[ST_MAXABS]) atomicMax((unsigned int *)&P.status[ST_MAXABS], mx);
        }
        *reinterpret_cast<int4 *>(&S.j[lane * 4]) = make_int4(0, 0, 0, 0);
        for (int i = lane; i <= nr && i <= NR_STAGE + 1; i += 32) S.off[i] = P.off[r_lo + i];
        for (int i = lane; i < nr && i <= NR_STAGE; i += 32) S.woff[i] = P.win_off[r_lo + i];
        __syncwarp();
        // ---- read boundaries: mark each later read's first call, then an inclusive max-scan
        for (int j = 1 + lane; j < nr; j += 32) {
            const long long o = (j <= NR_STAGE + 1 ? S.off[j] : P.off[r_lo + j]) - c0;
            if (o < len) atomicMax(&S.j[(int)o], j);
        }
        __syncwarp();
        {
            int4 v = *reinterpret_cast<int4 *>(&S.j[lane * 4]);
            v.y = max(v.x, v.y);
            v.z = max(v.y, v.z);
            v.w = max(v.z, v.w);
            int incl = v.w;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int o = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl = max(incl, o);
            }
            int excl = __shfl_up_sync(0xffffffffu, incl, 1);
            if (lane == 0) excl = 0;
            v.x = max(v.x, excl);
            v.y = max(v.y, excl);
            v.z = max(v.z, excl);
            v.w = max(v.w, excl);
            *reinterpret_cast<int4 *>(&S.j[lane * 4]) = v;
        }
        __syncwarp();

        // ---- windows (the pair that straddles two chunks is left to k_boundary_edges)
#pragma unroll 1
        for (int pl = lane; pl < len; pl += 32) {
            const bool halo = false;
            const int j = S.j[pl];
            const int64_t p = c0 + pl;
            const long long re = (j <= NR_STAGE) ? S.off[j + 1] : P.off[r_lo + j + 1];
            unsigned int val = INVALID_VAL;
            if (p + k <= re) {
                const int32_t *win = S.ids + pl;
                int dir = 0;
                unsigned long long klo = 0, khi = 0, h;
                if (K > 0) {
                    int g[K > 0 ? K : 1];
#pragma unroll
                    for (int i = 0; i < K; ++i) g[i] = win[i];
                    // window vs reverse complement, lexicographically: position i compares g[i] with
                    // -g[K-1-i]; positions past the middle repeat the first half's tests mirrored
#pragma unroll
                    for (int i = (K - 1) / 2; i >= 0; --i) {  // the first differing position decides
                        const int f = g[i], cc = -g[K - 1 - i];
                        if (f != cc) dir = f < cc ? 1 : -1;
                    }
                    if (packed && dir != 0) {
                        const unsigned int bias = 1u << (kb - 1);
#pragma unroll
                        for (int i = 0; i < K; ++i) {
                            const int cg = dir < 0 ? -g[K - 1 - i] : g[i];
                            khi = (khi << kb) | (klo >> (64 - kb));
                            klo = (klo << kb) | (unsigned long long)((unsigned int)cg + bias);
                        }
                    }
                } else {
                    for (int i = 0; i < k; ++i) {
                        const int f = win[i], cc = -win[k - 1 - i];
                        if (f != cc) {
                            dir = f < cc ? 1 : -1;
                            break;
                        }
                    }
                    if (packed && dir != 0) {
                        const unsigned int bias = 1u << (kb - 1);
                        for (int i = 0; i < k; ++i) {
                            const int cg = dir < 0 ? -win[k - 1 - i] : win[i];
                            khi = (khi << kb) | (klo >> (64 - kb));
                            klo = (klo << kb) | (unsigned long long)((unsigned int)cg + bias);
                        }
                    }
                }
                if (dir == 0) {
                    P.status[ST_ERR] = AMIRA_E_PALINDROME;  // construct_gene_mer.py:23-25
                } else {
                    const int dirneg = dir < 0;
                    h = packed ? (N16 ? (unsigned long long)packed_hash32(klo, khi) : packed_hash(klo, khi))
                               : canonical_hash(win, k, dirneg);
                    unsigned int slot;
                    if (N16) {
                        // the key's bits 63..84 take the place of the fingerprint
                        const unsigned long long top = (khi << 1) | (klo >> 63);
                        const unsigned long long mine =
                            (top << FP_SHIFT) | ((unsigned long long)p << 1) | (unsigned long long)dirneg;
                        slot = node_insert16(P, win, dirneg, klo & 0x7FFFFFFFFFFFFFFFull, h, mine);
                    } else {
                        const unsigned long long mine =
                            ((h >> FP_SHIFT) << FP_SHIFT) | ((unsigned long long)p << 1) | (unsigned long long)dirneg;
                        slot = node_insert(P, win, dirneg, packed, klo, khi, h, mine);
                    }
                    val = slot | ((unsigned int)dirneg << 31);
                    if (!halo) {
                        // Node.nodeCoverage: one per window (counts from 0xFFFFFFFF), fire and forget; it sizes the
                        // node's read list (incidence.cuh)
                        atomicAdd(N16 ? &P.ncov[slot] : &P.ntab[slot].cov, 1u);
                        const long long rs = (j <= NR_STAGE + 1) ? S.off[j] : P.off[r_lo + j];
                        const long long wo = (j <= NR_STAGE) ? S.woff[j] : P.win_off[r_lo + j];
                        const int64_t w = wo + (p - rs);
                        __stcs(&P.win_node[w], (int32_t)slot);  // streaming stores: keep the tables in L2
                        __stcs(&P.win_dir[w], (signed char)dir);
                        __stcs(&P.win_read[w], (int32_t)(P.read_base + r_lo + j));
                        if (P.ps) {
                            P.win_start[w] = __ldg(P.ps + p);
                            P.win_end[w] = __ldg(P.pe + p + k - 1);
                        }
                    }
                }
            }
            S.val[pl] = val;
        }
        __syncwarp();
        // ---- adjacent pairs of the same read
#define AMIRA_PAIR(pl_, valid_, key_, ord_)                                                                              \
    {                                                                                                                    \
        valid_ = false;                                                                                                  \
        key_ = 0;                                                                                                        \
        ord_ = 0;                                                                                                        \
        if ((pl_) + 1 < len) {                                                                                           \
            const unsigned int a_ = S.val[pl_], b_ = S.val[(pl_) + 1];                                                   \
            if (a_ != INVALID_VAL && b_ != INVALID_VAL && S.j[(pl_) + 1] == S.j[pl_]) {                                  \
                const unsigned int sa_ = a_ & 0x7FFFFFFFu, sb_ = b_ & 0x7FFFFFFFu;                                       \
                const unsigned int sdn_ = a_ >> 31, tdn_ = b_ >> 31;                                                     \
                key_ = ((unsigned long long)min(sa_, sb_) << 32) | ((unsigned long long)max(sa_, sb_) << 1) |            \
                       (unsigned long long)(sdn_ == tdn_);                                                               \
                ord_ = ((unsigned long long)(c0 + (pl_)) << 2) | ((unsigned long long)(sa_ > sb_) << 1) | sdn_;           \
                valid_ = true;                                                                                           \
            }                                                                                                            \
        }                                                                                                                \
    }
        if (E16) {
            // two pairs per lane in flight: both bucket loads are issued before either is looked at
#pragma unroll 1
            for (int pl = lane; pl + 1 < len; pl += 64) {
                bool v0, v1;
                unsigned long long k0, k1, r0, r1;
                AMIRA_PAIR(pl, v0, k0, r0);
                AMIRA_PAIR(pl + 32, v1, k1, r1);
                const unsigned int b0 = edge_bucket_of(P, k0), b1 = edge_bucket_of(P, k1);
                EdgeSlot16 *B0 = P.etab16 + 2 * (size_t)b0, *B1 = P.etab16 + 2 * (size_t)b1;
                unsigned long long x0 = 0, y0 = 0, x1 = 0, y1 = 0, u0 = 0, w0 = 0, u1 = 0, w1 = 0;
                if (v0) load_bucket(B0, x0, y0, x1, y1);
                if (v1) load_bucket(B1, u0, w0, u1, w1);
                if (v0 && !edge_bucket16(B0, k0, (unsigned int)r0, x0, y0, x1, y1)) edge_insert16_from(P, k0, (unsigned int)r0, b0 + 1);
                if (v1 && !edge_bucket16(B1, k1, (unsigned int)r1, u0, w0, u1, w1)) edge_insert16_from(P, k1, (unsigned int)r1, b1 + 1);
            }
        } else {
#pragma unroll 1
            for (int pl = lane; pl + 1 < len; pl += 32) {
                bool v0;
                unsigned long long k0, r0;
                AMIRA_PAIR(pl, v0, k0, r0);
                if (v0) edge_insert(P, k0, r0);
            }
        }
#undef AMIRA_PAIR
        __syncwarp();
    }
}

// The adjacent pair whose two windows start in different chunks (last call of chunk c-1, first call
// of chunk c): both windows were inserted by their own chunks, their slots are in win_node.
template <bool E16>
__global__ void k_boundary_edges(const BuildParams P) {
    const int64_t c = 1 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= P.n_tiles) return;
    const int64_t p1 = c * WC, p0 = p1 - 1;
    const int r = P.tile_r0[c];
    const int64_t rs = P.off[r], re = P.off[r + 1];
    if (rs > p0 || p1 + P.k > re) return;  // different reads, or no window starts at p1
    const int64_t w0 = P.win_off[r] + (p0 - rs);
    const unsigned int sa = (unsigned int)P.win_node[w0], sb = (unsigned int)P.win_node[w0 + 1];
    const unsigned int sdneg = P.win_dir[w0] < 0, tdneg = P.win_dir[w0 + 1] < 0;
    const unsigned int lo = min(sa, sb), hi = max(sa, sb);
    const unsigned long long key =
        ((unsigned long long)lo << 32) | ((unsigned long long)hi << 1) | (unsigned long long)(sdneg == tdneg);
    const unsigned long long ord = ((unsigned long long)p0 << 2) | ((unsigned long long)(sa > sb) << 1) | sdneg;
    if (E16) edge_insert16(P, key, (unsigned int)ord);
    else edge_insert(P, key, ord);
}

// ---------------------------------------------------------------------------------------------
// atomic roofline micro-benchmark: random-address RED.ADD.u32 / CAS.b64 into a table
__global__ void k_atomic_red(unsigned int *__restrict__ table, unsigned long long n_slots, unsigned long long n_ops,
                             unsigned long long seed) {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_ops; i += stride) {
        unsigned long long h = mix64(i + seed);
        atomicAdd(&table[(unsigned long long)(((h >> 32) * n_slots) >> 32) ], 1u);
    }
}

__global__ void k_atomic_cas(unsigned long long *__restrict__ table, unsigned long long n_slots,
                             unsigned long long n_ops, unsigned long long seed) {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long acc = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_ops; i += stride) {
        unsigned long long h = mix64(i + seed);
        acc += atomicCAS(&table[(unsigned long long)(((h >> 32) * n_slots) >> 32)], EMPTY64, h | 1ull);
    }
    if (acc == 0x123456789abcdefULL) table[0] = acc;  // keep the returns alive
}

// largest |id| of the input: decides how many bits a gene takes in the packed keys
__global__ void k_max_abs(const int32_t *__restrict__ ids, int64_t G, unsigned int *__restrict__ out) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned int m = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < G; i += stride) {
        const int g = __ldg(ids + i);
        m = max(m, (unsigned int)(g < 0 ? -(long long)g : (long long)g));
    }
    for (int d = 16; d > 0; d >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, d));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// random 32-byte sector loads (LDG.E.256 at L2), the other half of a hash-table probe
__global__ void k_random_load(const NodeSlot *__restrict__ table, unsigned long long n_slots, unsigned long long n_ops,
                              unsigned long long seed, unsigned long long *__restrict__ sink) {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long acc = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_ops; i += stride) {
        unsigned long long h = mix64(i + seed), a, b, c, d;
        load_node_slot(&table[(unsigned long long)(((h >> 32) * n_slots) >> 32)], a, b, c, d);
        acc += a ^ b ^ c ^ d;
    }
    if (acc == 0x123456789abcdefULL) *sink = acc;
}

}  // namespace amira
