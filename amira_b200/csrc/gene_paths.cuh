// gene_paths.cuh -- the reads grouped by their path through the genes of interest (amira_gmg_gene_paths), over the
// per-read windows of the gene-mer graph (win_off / win_node / win_dir) and the marked nodes of k_nodes_containing.
//
// A window is live when win_node >= 0; its state is window_state (unitigs.cuh).  An occurrence is a maximal run of
// live windows on marked nodes within one read; its span adds the live window on each side (the flanks), and its key
// is the smaller of the span's state sequence S and its mirror R(S) (reversed, every state ^ 1).
//
//  - k_gp_flags: one thread per window flags "starts a run" and "ends a run".
//  - one scan over the W flags numbers the occurrences in window order (GpOccStore writes occ_read, occ_win and the
//    run's end, which k_gp_span turns into its length).  The scan runs once to count and once to write, so the
//    per-occurrence arrays are sized by the count, not by W.
//  - k_gp_span: one thread per occurrence finds the flanks, compares S with R(S) from both ends, and hashes the
//    canonical sequence (64 bits, or a few with the test hook, so that every probe compares sequences).
//  - k_gp_group: one thread per complete occurrence probes an open-addressing table (a power of two, at least twice
//    the complete occurrences) by the hash.  A slot holds the first occurrence that claimed it; on a hash match the two
//    canonical sequences are compared through the windows.  atomicMin keeps the smallest occurrence of every slot.
//  - one scan over "is the first of its slot" numbers the clusters in first-occurrence order (GpClusterStore);
//    k_gp_cluster gives every complete occurrence its cluster.
//  - one scan over the key lengths gives key_off; k_gp_key_fill writes each cluster's key and counts its states per
//    node; a scan over the N nodes gives the containment index's offsets, and k_gp_key_place fills it with (cluster,
//    position) entries.
//  - k_gp_match: one thread per partial occurrence walks the entries of the node of its first state and tests both
//    alignments (S at the entry, or R(S) ending at it), keeping the first cluster seen and whether another was seen.
//    Cost: O(partials x entries of that node x span length).
//  - k_gp_member_count / a scan / k_gp_member_place fill the members of every cluster (cursor atomics); the segmented
//    sort of segsort.cuh then orders each cluster's members ascending.
#pragma once

#include "correct.cuh"
#include "segsort.cuh"

namespace amira {

constexpr uint8_t GP_START = 1, GP_END = 2;
constexpr uint8_t GP_LEFT = 1, GP_RIGHT = 2;
constexpr uint32_t GP_EMPTY = 0xFFFFFFFFu;

__device__ __forceinline__ bool gp_marked(const int32_t *__restrict__ win_node, const uint8_t *__restrict__ marked,
                                          const long long w) {
    const int32_t n = win_node[w];
    return n >= 0 && marked[n];
}

__global__ void k_gp_flags(const int32_t *__restrict__ win_node, const int32_t *__restrict__ win_read, const long long W,
                           const uint8_t *__restrict__ marked, uint8_t *__restrict__ flags) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    if (!gp_marked(win_node, marked, w)) {
        flags[w] = 0;
        return;
    }
    const int32_t r = win_read[w];
    const bool in = w > 0 && win_read[w - 1] == r && gp_marked(win_node, marked, w - 1);
    const bool out = w + 1 < W && win_read[w + 1] == r && gp_marked(win_node, marked, w + 1);
    flags[w] = (in ? 0 : GP_START) | (out ? 0 : GP_END);
}

struct GpOccLoad {
    const uint8_t *flags;
    __device__ __forceinline__ unsigned long long operator()(long long w) const { return flags[w] & GP_START; }
};
// ... -> at a run's start occ_read / occ_win, at its end occ_length = the end within its read (k_gp_span subtracts
// occ_win); *n_occ = the occurrences.  occ_read == nullptr: the count only.
struct GpOccStore {
    const uint8_t *flags;
    const int32_t *win_read;
    const int64_t *win_off;
    long long W;
    int32_t *occ_read, *occ_win, *occ_length;
    unsigned long long *n_occ;
    __device__ __forceinline__ void operator()(long long w, unsigned long long excl, unsigned long long start) const {
        if (w == W) {
            *n_occ = excl;
            return;
        }
        const uint8_t f = flags[w];
        if (!f || !occ_read) return;
        const int32_t r = win_read[w];
        const long long first = win_off[r];
        if (start) {
            occ_read[excl] = r;
            occ_win[excl] = (int32_t)(w - first);
        }
        if (f & GP_END) occ_length[excl + start - 1] = (int32_t)(w + 1 - first);
    }
};

// the span of occurrence o: its first window (global index) and its length
struct GpSpans {
    const int64_t *span_w;
    const int32_t *span_len;
    const int8_t *orient;
    const int32_t *win_node;
    const int8_t *win_dir;
    __device__ __forceinline__ int32_t state(const long long w) const { return window_state(win_node[w], win_dir[w]); }
    // element t of o's canonical sequence
    __device__ __forceinline__ int32_t canon(const long long o, const int32_t t) const {
        const long long w0 = span_w[o];
        return orient[o] > 0 ? state(w0 + t) : state(w0 + span_len[o] - 1 - t) ^ 1;
    }
    __device__ __forceinline__ bool same_key(const long long a, const long long b) const {
        const int32_t L = span_len[a];
        if (span_len[b] != L) return false;
        for (int32_t t = 0; t < L; ++t)
            if (canon(a, t) != canon(b, t)) return false;
        return true;
    }
};

__device__ __forceinline__ unsigned long long gp_mix(unsigned long long x) {
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebull;
    x ^= x >> 31;
    return x;
}

// one thread per occurrence: flanks, span, orientation (ties +1) and the hash of the canonical sequence
__global__ void k_gp_span(const int32_t *__restrict__ occ_read, const int32_t *__restrict__ occ_win,
                          int32_t *__restrict__ occ_length, const long long O, const int64_t *__restrict__ win_off,
                          const int32_t *__restrict__ win_node, const int8_t *__restrict__ win_dir, const int hash_bits,
                          uint8_t *__restrict__ occ_flanks, int8_t *__restrict__ occ_orient, int64_t *__restrict__ span_w,
                          int32_t *__restrict__ span_len, unsigned long long *__restrict__ occ_hash) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= O) return;
    const int32_t r = occ_read[o], i = occ_win[o], len = occ_length[o] - i;
    occ_length[o] = len;
    const long long w0 = win_off[r], nw = win_off[r + 1] - w0;
    const bool left = i >= 1 && win_node[w0 + i - 1] >= 0;
    const bool right = i + len < nw && win_node[w0 + i + len] >= 0;
    occ_flanks[o] = (left ? GP_LEFT : 0) | (right ? GP_RIGHT : 0);
    const long long s0 = w0 + i - (left ? 1 : 0);
    const int32_t L = len + (left ? 1 : 0) + (right ? 1 : 0);
    span_w[o] = s0;
    span_len[o] = L;
    // S[t] against R(S)[t] = S[L - 1 - t] ^ 1 up to the middle (which differs from its own mirror); a tie is +1
    int8_t orient = 1;
    for (int32_t t = 0; t <= L - 1 - t; ++t) {
        const int32_t a = window_state(win_node[s0 + t], win_dir[s0 + t]);
        const int32_t b = window_state(win_node[s0 + L - 1 - t], win_dir[s0 + L - 1 - t]) ^ 1;
        if (a != b) {
            orient = a < b ? 1 : -1;
            break;
        }
    }
    occ_orient[o] = orient;
    unsigned long long h = gp_mix(0x9e3779b97f4a7c15ull + (unsigned long long)L);
    for (int32_t t = 0; t < L; ++t) {
        const long long w = orient > 0 ? s0 + t : s0 + L - 1 - t;
        const int32_t s = window_state(win_node[w], win_dir[w]) ^ (orient > 0 ? 0 : 1);
        h = gp_mix(h ^ (unsigned long long)(uint32_t)s);
    }
    occ_hash[o] = hash_bits < 64 ? (h & ((1ull << hash_bits) - 1ull)) : h;
}

// one thread per complete occurrence: the slot of its key (probed by hash, sequences compared on a hash match), and
// the smallest occurrence of every slot
__global__ void k_gp_group(const uint8_t *__restrict__ occ_flanks, const unsigned long long *__restrict__ occ_hash,
                           const long long O, const GpSpans sp, const unsigned long long mask,
                           uint32_t *__restrict__ slot_occ, uint32_t *__restrict__ slot_first, uint32_t *__restrict__ occ_slot) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= O || occ_flanks[o] != (GP_LEFT | GP_RIGHT)) return;
    const unsigned long long h = occ_hash[o];
    unsigned long long i = gp_mix(h) & mask;
    while (true) {
        uint32_t v = slot_occ[i];
        if (v == GP_EMPTY) {
            v = atomicCAS(&slot_occ[i], GP_EMPTY, (uint32_t)o);
            if (v == GP_EMPTY) break;
        }
        if (occ_hash[v] == h && sp.same_key(v, o)) break;
        i = (i + 1) & mask;
    }
    occ_slot[o] = (uint32_t)i;
    atomicMin(&slot_first[i], (uint32_t)o);
}

struct GpFirstLoad {
    const uint8_t *occ_flanks;
    const uint32_t *occ_slot, *slot_first;
    __device__ __forceinline__ unsigned long long operator()(long long o) const {
        return occ_flanks[o] == (GP_LEFT | GP_RIGHT) && slot_first[occ_slot[o]] == (uint32_t)o;
    }
};
// ... -> a first occurrence gets cluster excl (occ_cluster, cluster_first, key_len); *n_clusters
struct GpClusterStore {
    long long O;
    const int32_t *span_len;
    int32_t *occ_cluster;
    uint32_t *cluster_first, *key_len;
    unsigned long long *n_clusters;
    __device__ __forceinline__ void operator()(long long o, unsigned long long excl, unsigned long long first) const {
        if (o == O) *n_clusters = excl;
        else if (first) {
            occ_cluster[o] = (int32_t)excl;
            cluster_first[excl] = (uint32_t)o;
            key_len[excl] = (uint32_t)span_len[o];
        }
    }
};

__global__ void k_gp_cluster(const uint8_t *__restrict__ occ_flanks, const uint32_t *__restrict__ occ_slot,
                             const uint32_t *__restrict__ slot_first, const long long O, int32_t *__restrict__ occ_cluster) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= O || occ_flanks[o] != (GP_LEFT | GP_RIGHT)) return;
    const uint32_t f = slot_first[occ_slot[o]];
    if (f != (uint32_t)o) occ_cluster[o] = occ_cluster[f];
}

// offsets from a scan over counts, and a copy as the cursor of the placement (nullable)
struct GpOffStore {
    int64_t *off;
    unsigned long long *cursor;
    __device__ __forceinline__ void operator()(long long i, unsigned long long excl, unsigned long long) const {
        off[i] = (int64_t)excl;
        if (cursor) cursor[i] = excl;
    }
};

// one thread per cluster: its key (the canonical sequence of its first occurrence) and its states counted per node
__global__ void k_gp_key_fill(const uint32_t *__restrict__ cluster_first, const long long C, const int64_t *__restrict__ key_off,
                              const GpSpans sp, int32_t *__restrict__ key_state, unsigned long long *__restrict__ node_cnt) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const long long o = cluster_first[c], k0 = key_off[c];
    const int32_t L = (int32_t)(key_off[c + 1] - k0);
    for (int32_t t = 0; t < L; ++t) {
        const int32_t s = sp.canon(o, t);
        key_state[k0 + t] = s;
        atomicAdd(&node_cnt[s >> 1], 1ull);
    }
}

__global__ void k_gp_key_place(const long long C, const int64_t *__restrict__ key_off, const int32_t *__restrict__ key_state,
                               unsigned long long *__restrict__ cursor, int32_t *__restrict__ ent_cluster,
                               int32_t *__restrict__ ent_pos) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const long long k0 = key_off[c];
    const int32_t L = (int32_t)(key_off[c + 1] - k0);
    for (int32_t t = 0; t < L; ++t) {
        const unsigned long long e = atomicAdd(&cursor[key_state[k0 + t] >> 1], 1ull);
        ent_cluster[e] = (int32_t)c;
        ent_pos[e] = t;
    }
}

// one thread per partial occurrence: the clusters whose key holds S or R(S), through the entries of the node of S[0]
__global__ void k_gp_match(const uint8_t *__restrict__ occ_flanks, const long long O, const int64_t *__restrict__ span_w,
                           const int32_t *__restrict__ span_len, const int32_t *__restrict__ win_node,
                           const int8_t *__restrict__ win_dir, const int64_t *__restrict__ node_off,
                           const int32_t *__restrict__ ent_cluster, const int32_t *__restrict__ ent_pos,
                           const int64_t *__restrict__ key_off, const int32_t *__restrict__ key_state,
                           int32_t *__restrict__ occ_cluster, int8_t *__restrict__ occ_orient) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= O || occ_flanks[o] == (GP_LEFT | GP_RIGHT)) return;
    const long long s0 = span_w[o];
    const int32_t L = span_len[o];
    const int32_t first = window_state(win_node[s0], win_dir[s0]);
    int32_t c1 = -1;
    bool fwd = false, multi = false;
    for (long long e = node_off[first >> 1]; e < node_off[(first >> 1) + 1] && !multi; ++e) {
        const int32_t c = ent_cluster[e], j = ent_pos[e];
        const int64_t k0 = key_off[c];
        const int32_t kl = (int32_t)(key_off[c + 1] - k0);
        const int32_t *key = key_state + k0;
        bool hit = false, forward = false;
        if (key[j] == first) {  // S at j
            if (j + L <= kl) {
                hit = true;
                for (int32_t t = 1; t < L && hit; ++t) hit = key[j + t] == window_state(win_node[s0 + t], win_dir[s0 + t]);
                forward = hit;
            }
        } else if (j - (L - 1) >= 0) {  // key[j] == first ^ 1: R(S) ends at j
            hit = true;
            const int32_t b = j - (L - 1);
            for (int32_t t = 0; t < L - 1 && hit; ++t)
                hit = key[b + t] == (window_state(win_node[s0 + L - 1 - t], win_dir[s0 + L - 1 - t]) ^ 1);
        }
        if (!hit) continue;
        if (c1 < 0) c1 = c;
        else if (c != c1) multi = true;
        if (c == c1 && forward) fwd = true;
    }
    if (multi) occ_cluster[o] = -2;
    else if (c1 < 0) occ_cluster[o] = -1;
    else {
        occ_cluster[o] = c1;
        occ_orient[o] = fwd ? 1 : -1;
    }
}

// members: the occurrences with a cluster, counted per cluster (and the complete ones), then placed
__global__ void k_gp_member_count(const int32_t *__restrict__ occ_cluster, const uint8_t *__restrict__ occ_flanks,
                                  const long long O, uint32_t *__restrict__ member_cnt, uint32_t *__restrict__ n_complete) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= O) return;
    const int32_t c = occ_cluster[o];
    if (c < 0) return;
    atomicAdd(&member_cnt[c], 1u);
    if (occ_flanks[o] == (GP_LEFT | GP_RIGHT)) atomicAdd(&n_complete[c], 1u);
}

__global__ void k_gp_member_place(const int32_t *__restrict__ occ_cluster, const long long O,
                                  unsigned long long *__restrict__ cursor, uint32_t *__restrict__ members) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= O) return;
    const int32_t c = occ_cluster[o];
    if (c >= 0) members[atomicAdd(&cursor[c], 1ull)] = (uint32_t)o;
}

}  // namespace amira
