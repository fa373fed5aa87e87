// bubbles.cuh -- the simple bubbles of the compacted graph (amira_gmg_bubbles), over the cached unitigs (unitigs.cuh)
// and read paths.
//
// A state is s = 2 * node + side; list(s) is that node's forward (side 0) or backward (side 1) list.  A directed edge
// e = (u -> v, sd, td) lies in list(2u + (sd < 0)) and continues through cont(e) = 2v + (td < 0); v's entering list
// for e is list(cont(e) ^ 1).  e in list(sigma), x = sigma >> 1, h = v, enters a branch b (the unitig of h) when
// list(cont(e) ^ 1) holds one edge, b is not circular, the walk through b from h in the direction of cont(e) ends
// at b's other end t, left through s_t, list(s_t) holds one edge e' (target y), and neither x nor y is a node of b.
// The branch runs from sigma to tau = cont(e').  Branches of one list with the same tau form a bubble when there are
// two or more of them and sigma < (tau ^ 1); the mirror (from tau ^ 1 to sigma ^ 1) is not reported.
//
//  - k_bubble_branches: one thread per directed edge evaluates the conditions and writes tau when the edge enters a
//    branch of the canonical orientation (sigma < tau ^ 1), -1 otherwise.  The walk through b is a lookup: when x is
//    not in b, h is b's end on the entering side (its one-edge entering list holds the reverse of e, so no state of
//    b precedes it), t is the other end in listed order, and s_t is t's listed state (flipped when b is walked
//    against its listed order).  An edge with x in b fails condition 4 whatever t is.
//  - k_bubble_group: one warp per 32 states.  A state whose list holds fewer than two edges is done by its own lane;
//    the warp then takes the other states one at a time and groups their list entries by tau in tiles of 32: per
//    entry the number of entries with its tau, how many come before it, and the first of them (one broadcast per
//    entry of every tile: O(d^2 / 32) warp steps for a list of d edges); then per entry the branches of the groups
//    whose first entry comes before its group's.  It writes per edge its branch and bubble number within the list,
//    and per state its bubble and branch counts packed into one 64-bit word (bubbles << 32 | branches: B < 2^30 and
//    the branches < 2^31, so a scan of the packed words sums both without a carry).
//  - one scan over the 2N states gives each state's first bubble and branch, and the totals (branch_off[B]).
//  - k_bubble_fill: one thread per edge in a bubble writes its branch (unitig, orientation, the unitig -> branch
//    map), and the first edge of every bubble writes the bubble (source, sink, first branch).
//  - k_bubble_reads: one thread per read step adds 1 (integer atomics) to the branch of its unitig when the step is
//    as long as the unitig.
// Ordering comes from the list positions alone, never from thread timing: bubbles by sigma, then by the list
// position of their first branch; branches by list position.
//
// The popping policy (amira_gmg_bubble_policy) over the cached bubbles and unitigs:
//  - k_bubble_spare: one thread per node flagged as holding a gene of interest marks the branch of its unitig spared.
//  - k_bubble_policy: one warp per bubble finds the kept branch (largest mean node coverage, compared exactly; then
//    most branch_reads; then lowest index) and writes replace_with for every branch of the bubble.
#pragma once

#include "unitigs.cuh"

namespace amira {

// the single edge of list(s), which must hold exactly one
__device__ __forceinline__ uint32_t adj_only_edge(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges,
                                                  const long long N, const int32_t s) {
    return adj_edges[adj_off[(s & 1) * N + (s >> 1)]];
}

__global__ void k_bubble_branches(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges, const long long N,
                                  const int32_t *__restrict__ e_src, const int32_t *__restrict__ e_tgt,
                                  const int8_t *__restrict__ e_sd, const int8_t *__restrict__ e_td, const long long E,
                                  const int32_t *__restrict__ node_unitig, const int8_t *__restrict__ node_orient,
                                  const int64_t *__restrict__ unitig_off, const int32_t *__restrict__ unitig_nodes,
                                  const uint8_t *__restrict__ circular, int32_t *__restrict__ edge_tau) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= E) return;
    int32_t tau = -1;
    const int32_t x = e_src[j], v = e_tgt[j];
    const int32_t sigma = 2 * x + (e_sd[j] < 0 ? 1 : 0), c = 2 * v + (e_td[j] < 0 ? 1 : 0);
    const int32_t b = node_unitig[v];
    if (adj_list_size(adj_off, N, c >> 1, (c & 1) ^ 1) == 1 && !circular[b]) {
        const bool along = c == 2 * v + (node_orient[v] < 0 ? 1 : 0);  // the walk follows b's listed order
        const int32_t t = along ? unitig_nodes[unitig_off[b + 1] - 1] : unitig_nodes[unitig_off[b]];
        const int32_t st = (2 * t + (node_orient[t] < 0 ? 1 : 0)) ^ (along ? 0 : 1);
        if (adj_list_size(adj_off, N, t, st & 1) == 1) {
            const uint32_t e2 = adj_only_edge(adj_off, adj_edges, N, st);
            const int32_t y = e_tgt[e2];
            const int32_t t2 = 2 * y + (e_td[e2] < 0 ? 1 : 0);
            if (node_unitig[x] != b && node_unitig[y] != b && sigma < (t2 ^ 1)) tau = t2;
        }
    }
    edge_tau[j] = tau;
}

// per edge: ebr = its branch number within its list (-1: in no bubble), ebub = its bubble number within the list when
// it is the bubble's first branch (-1 otherwise), ehead = scratch; per state: (bubbles << 32) | branches
__global__ void k_bubble_group(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges, const long long N,
                               const int32_t *__restrict__ edge_tau, int32_t *__restrict__ ebr, int32_t *__restrict__ ebub,
                               int32_t *__restrict__ ehead, unsigned long long *__restrict__ counts) {
    const int lane = threadIdx.x & 31;
    const long long s0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) & ~31ll, S = 2 * N;
    const long long s = s0 + lane;
    long long d = 0;
    if (s < S) {
        const long long lo = adj_off[(s & 1) * N + (s >> 1)];
        d = adj_off[(s & 1) * N + (s >> 1) + 1] - lo;
        if (d < 2) {
            counts[s] = 0ull;
            if (d == 1) {
                const uint32_t j = adj_edges[lo];
                ebr[j] = -1;
                ebub[j] = -1;
            }
        }
    }
    unsigned many = __ballot_sync(0xffffffffu, d >= 2);
    while (many) {
        const int src_lane = __ffs(many) - 1;
        many &= many - 1;
        const long long sg = s0 + src_lane;
        const long long lo = adj_off[(sg & 1) * N + (sg >> 1)];
        const long long dd = adj_off[(sg & 1) * N + (sg >> 1) + 1] - lo;
        // pass 1: per entry its group size, entries of its group before it, and its group's first entry
        for (long long a = 0; a < dd; a += 32) {
            const long long i = a + lane;
            const uint32_t j = i < dd ? adj_edges[lo + i] : 0u;
            const int32_t ki = i < dd ? edge_tau[j] : -1;
            int cnt = 0, before = 0;
            long long first = i;
            for (long long b = 0; b < dd; b += 32) {
                const int32_t kb = b + lane < dd ? edge_tau[adj_edges[lo + b + lane]] : -1;
                const int last = (int)min(32ll, dd - b);
                for (int l = 0; l < last; ++l) {
                    const int32_t k = __shfl_sync(0xffffffffu, kb, l);
                    if (ki >= 0 && k == ki) {
                        ++cnt;
                        if (b + l < i) ++before;
                        first = min(first, b + l);
                    }
                }
            }
            if (i < dd) {
                const bool in = ki >= 0 && cnt >= 2;
                ehead[j] = in && before == 0 ? cnt : 0;
                ebr[j] = in ? before : -1;
                ebub[j] = in ? (int32_t)first : -1;
            }
        }
        __syncwarp();
        // pass 2: the branches and bubbles of the groups whose first entry comes before this entry's group's
        int n_bub = 0, n_br = 0;
        for (long long a = 0; a < dd; a += 32) {
            const long long i = a + lane;
            const uint32_t j = i < dd ? adj_edges[lo + i] : 0u;
            const int32_t mine = i < dd ? ebr[j] : -1;
            const long long first = mine >= 0 ? (long long)ebub[j] : -1;
            int br = 0, bub = 0;
            for (long long b = 0; b < dd; b += 32) {
                const int32_t hb = b + lane < dd ? ehead[adj_edges[lo + b + lane]] : 0;
                const int last = (int)min(32ll, dd - b);
                for (int l = 0; l < last; ++l) {
                    const int32_t c = __shfl_sync(0xffffffffu, hb, l);
                    if (c > 0 && b + l < first) {
                        br += c;
                        ++bub;
                    }
                }
            }
            if (mine >= 0) {
                ebr[j] = br + mine;
                ebub[j] = mine == 0 ? bub : -1;
            }
            n_bub += __popc(__ballot_sync(0xffffffffu, mine == 0));
            n_br += __popc(__ballot_sync(0xffffffffu, mine >= 0));
        }
        if (lane == 0) counts[sg] = ((unsigned long long)n_bub << 32) | (unsigned long long)n_br;
        __syncwarp();
    }
}

struct BubbleCountLoad {
    const unsigned long long *counts;
    __device__ __forceinline__ unsigned long long operator()(long long s) const { return counts[s]; }
};
// ... -> first[s] = (first bubble << 32) | first branch of state s; totals -> *n_out, branch_off[B] = branches
struct BubbleCountStore {
    unsigned long long *first;
    long long S;
    unsigned long long *n_out;
    int64_t *branch_off;
    __device__ __forceinline__ void operator()(long long s, unsigned long long excl, unsigned long long) const {
        if (s == S) {
            *n_out = excl;
            branch_off[excl >> 32] = (int64_t)(excl & 0xffffffffull);
        } else {
            first[s] = excl;
        }
    }
};

__global__ void k_bubble_fill(const int32_t *__restrict__ ebr, const int32_t *__restrict__ ebub, const int32_t *__restrict__ edge_tau,
                              const long long E, const int32_t *__restrict__ e_src, const int32_t *__restrict__ e_tgt,
                              const int8_t *__restrict__ e_sd, const unsigned long long *__restrict__ first,
                              const int32_t *__restrict__ node_unitig, const int64_t *__restrict__ unitig_off,
                              const int32_t *__restrict__ unitig_nodes, int32_t *__restrict__ source, int32_t *__restrict__ sink,
                              int64_t *__restrict__ branch_off, int32_t *__restrict__ branch_unitig,
                              int8_t *__restrict__ branch_orient, int32_t *__restrict__ unitig_branch) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= E) return;
    const int32_t r = ebr[j];
    if (r < 0) return;
    const int32_t sigma = 2 * e_src[j] + (e_sd[j] < 0 ? 1 : 0), v = e_tgt[j], b = node_unitig[v];
    const unsigned long long f = first[sigma];
    const long long g = (long long)(f & 0xffffffffull) + r;
    branch_unitig[g] = b;
    branch_orient[g] = (int8_t)(unitig_nodes[unitig_off[b]] == v ? 1 : -1);
    unitig_branch[b] = (int32_t)g;
    const int32_t q = ebub[j];
    if (q >= 0) {
        const long long i = (long long)(f >> 32) + q;
        source[i] = sigma;
        sink[i] = edge_tau[j];
        branch_off[i] = g;
    }
}

__global__ void k_bubble_reads(const int32_t *__restrict__ step_unitig, const int32_t *__restrict__ step_length, const long long T,
                               const int32_t *__restrict__ unitig_branch, const int64_t *__restrict__ unitig_off,
                               uint32_t *__restrict__ branch_reads) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const int32_t b = step_unitig[t], g = unitig_branch[b];
    if (g >= 0 && (int64_t)step_length[t] == unitig_off[b + 1] - unitig_off[b]) atomicAdd(&branch_reads[g], 1u);
}

// ---- the popping policy (amira_gmg_bubble_policy) ----------------------------------------------------------------

// one thread per node: a node flagged by k_nodes_containing spares the branch its unitig is (plain stores of 1)
__global__ void k_bubble_spare(const uint8_t *__restrict__ flags, const long long N, const int32_t *__restrict__ node_unitig,
                               const int32_t *__restrict__ unitig_branch, uint8_t *__restrict__ spared) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N || !flags[n]) return;
    const int32_t g = unitig_branch[node_unitig[n]];
    if (g >= 0) spared[g] = 1;
}

// a branch's rank key: mean node coverage cs / ln, then reads, then (lower first) its index
struct BranchRank {
    unsigned long long cs, ln;
    uint32_t rd;
    int32_t g;  // -1: no branch
};

// a beats b.  The means are compared as cs_a * ln_b against cs_b * ln_a, exactly, in 128 bits: cs is a sum of 32-bit
// coverages over up to 2^30 nodes (< 2^62) and ln < 2^31, so the products need up to 93 bits.
__device__ __forceinline__ bool branch_beats(const BranchRank &a, const BranchRank &b) {
    if (b.g < 0) return a.g >= 0;
    if (a.g < 0) return false;
    const unsigned long long lh = __umul64hi(a.cs, b.ln), rh = __umul64hi(b.cs, a.ln);
    if (lh != rh) return lh > rh;
    const unsigned long long ll = a.cs * b.ln, rl = b.cs * a.ln;
    if (ll != rl) return ll > rl;
    if (a.rd != b.rd) return a.rd > b.rd;
    return a.g < b.g;
}

// one warp per bubble, strided over its branches (a bubble may have any number): each lane keeps the best of its
// branches, a butterfly of shuffles leaves the bubble's winner in every lane, then every branch that is not the winner
// and not spared gets replace[g] = winner, others -1.  The replaced branches are counted with a ballot per stride and
// one atomic per warp.
__global__ void k_bubble_policy(const int64_t *__restrict__ branch_off, const long long B, const int32_t *__restrict__ branch_unitig,
                                const uint32_t *__restrict__ branch_reads, const int64_t *__restrict__ unitig_off,
                                const unsigned long long *__restrict__ cov_sum, const uint8_t *__restrict__ spared,
                                int32_t *__restrict__ replace, unsigned long long *__restrict__ n_replaced) {
    const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q >= B) return;  // whole warps: B is per warp
    const long long lo = branch_off[q], hi = branch_off[q + 1];
    BranchRank best{0, 0, 0, -1};
    for (long long g = lo + lane; g < hi; g += 32) {
        const int32_t b = branch_unitig[g];
        const BranchRank x{cov_sum[b], (unsigned long long)(unitig_off[b + 1] - unitig_off[b]), branch_reads[g], (int32_t)g};
        if (branch_beats(x, best)) best = x;
    }
    for (int d = 16; d > 0; d >>= 1) {
        BranchRank o;
        o.cs = __shfl_xor_sync(0xffffffffu, best.cs, d);
        o.ln = __shfl_xor_sync(0xffffffffu, best.ln, d);
        o.rd = __shfl_xor_sync(0xffffffffu, best.rd, d);
        o.g = __shfl_xor_sync(0xffffffffu, best.g, d);
        if (branch_beats(o, best)) best = o;
    }
    unsigned int count = 0;
    for (long long base = lo; base < hi; base += 32) {
        const long long g = base + lane;
        const bool rep = g < hi && g != best.g && !spared[g];
        if (g < hi) replace[g] = rep ? best.g : -1;
        count += __popc(__ballot_sync(0xffffffffu, rep));
    }
    if (lane == 0 && count) atomicAdd(n_replaced, (unsigned long long)count);
}

}  // namespace amira
