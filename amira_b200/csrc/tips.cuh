// tips.cuh -- the dead-end tips of the compacted graph (amira_gmg_tips), the clipping policy (amira_gmg_tip_policy) and
// the reads clipped at them (amira_gmg_clip_tip_reads), over the cached unitigs and read paths (unitigs.cuh).
//
// States, lists and cont(e) as in bubbles.cuh.  A non-circular unitig b with first node h0 and last node h1 (listed
// order) has two outward end states: out1 = 2 * h1 + (node_orient[h1] < 0) and out0 = (2 * h0 + (node_orient[h0] < 0))
// ^ 1.  b is a tip when exactly one of list(out0), list(out1) is empty and the other, list(s_t), holds exactly one edge
// e' whose target v is not a node of b.  attach = cont(e') ^ 1 (v's list that holds the edge into b), orient = +1 when
// the dead end is out1 (a walk from v into b follows the listed order).
//
//  - k_tip_flags: one thread per unitig tests the tip condition.
//  - one scan over the U flags numbers the tips (TipStore writes tip_unitig[q] = b and the count).
//  - k_tip_fill: one thread per tip writes its orientation and attach state, and unitig_tip[b] = q.
//  - k_tip_reads: one thread per read step adds 1 (integer atomics) to the tip of its unitig.
//
// The policy: k_bubble_spare (bubbles.cuh) over unitig_tip marks the tips with a node holding a gene of interest;
// k_tip_policy, one warp per tip, strides over list(attach) and clips the tip when it is short, not spared, and some
// edge of the list leads into another unitig with a strictly larger mean node coverage (exact 128-bit cross
// products).  A list of d edges costs O(d) per tip, so O(d^2) over d tips that share it.
//
// The clip: k_tip_clip, one thread per read step on a clipped tip, marks the calls it drops with code 1 in the
// correction's cnt array (correct.cuh: 0 untouched, 1 no output call), flags the read and counts the tip.  The scan,
// k_correct_offsets and k_correct_fill of correct.cuh then write the clipped CSR; they never read the step fields for
// codes 0 and 1.
#pragma once

#include "correct.cuh"

namespace amira {

// the state a walk leaves node n through in its unitig's listed order
__device__ __forceinline__ int32_t listed_state(const int8_t *__restrict__ node_orient, const int32_t n) {
    return 2 * n + (node_orient[n] < 0 ? 1 : 0);
}

// 1 when unitig b is a tip; *st = its attached end state s_t (the one-edge list), *dead1 = the dead end is out1
__device__ __forceinline__ bool tip_ends(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges,
                                         const long long N, const int32_t *__restrict__ e_tgt,
                                         const int32_t *__restrict__ node_unitig, const int8_t *__restrict__ node_orient,
                                         const int64_t *__restrict__ unitig_off, const int32_t *__restrict__ unitig_nodes,
                                         const int32_t b, int32_t *st, bool *dead1) {
    const int32_t h0 = unitig_nodes[unitig_off[b]], h1 = unitig_nodes[unitig_off[b + 1] - 1];
    const int32_t out1 = listed_state(node_orient, h1), out0 = listed_state(node_orient, h0) ^ 1;
    const long long d0 = adj_list_size(adj_off, N, out0 >> 1, out0 & 1), d1 = adj_list_size(adj_off, N, out1 >> 1, out1 & 1);
    if (!((d0 == 0 && d1 == 1) || (d1 == 0 && d0 == 1))) return false;
    *dead1 = d1 == 0;
    *st = *dead1 ? out0 : out1;
    return node_unitig[e_tgt[adj_only_edge(adj_off, adj_edges, N, *st)]] != b;
}

__global__ void k_tip_flags(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges, const long long N,
                            const int32_t *__restrict__ e_tgt, const int32_t *__restrict__ node_unitig,
                            const int8_t *__restrict__ node_orient, const int64_t *__restrict__ unitig_off,
                            const int32_t *__restrict__ unitig_nodes, const uint8_t *__restrict__ circular, const long long U,
                            uint8_t *__restrict__ flags) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= U) return;
    int32_t st;
    bool dead1;
    flags[b] = !circular[b] && tip_ends(adj_off, adj_edges, N, e_tgt, node_unitig, node_orient, unitig_off, unitig_nodes,
                                        (int32_t)b, &st, &dead1);
}

struct TipLoad {
    const uint8_t *flags;
    __device__ __forceinline__ unsigned long long operator()(long long b) const { return flags[b]; }
};
// ... -> tip_unitig[excl] = b for a tip; *n_tips = the tips
struct TipStore {
    int32_t *tip_unitig;
    long long U;
    unsigned long long *n_tips;
    __device__ __forceinline__ void operator()(long long b, unsigned long long excl, unsigned long long tip) const {
        if (b == U) *n_tips = excl;
        else if (tip) tip_unitig[excl] = (int32_t)b;
    }
};

__global__ void k_tip_fill(const int32_t *__restrict__ tip_unitig, const long long Q, const int64_t *__restrict__ adj_off,
                           const uint32_t *__restrict__ adj_edges, const long long N, const int32_t *__restrict__ e_tgt,
                           const int8_t *__restrict__ e_td, const int32_t *__restrict__ node_unitig,
                           const int8_t *__restrict__ node_orient, const int64_t *__restrict__ unitig_off,
                           const int32_t *__restrict__ unitig_nodes, int8_t *__restrict__ tip_orient,
                           int32_t *__restrict__ tip_attach, int32_t *__restrict__ unitig_tip) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    const int32_t b = tip_unitig[q];
    int32_t st;
    bool dead1;
    tip_ends(adj_off, adj_edges, N, e_tgt, node_unitig, node_orient, unitig_off, unitig_nodes, b, &st, &dead1);
    const uint32_t e = adj_only_edge(adj_off, adj_edges, N, st);
    tip_orient[q] = dead1 ? 1 : -1;
    tip_attach[q] = (2 * e_tgt[e] + (e_td[e] < 0 ? 1 : 0)) ^ 1;
    unitig_tip[b] = (int32_t)q;
}

__global__ void k_tip_reads(const int32_t *__restrict__ step_unitig, const long long T, const int32_t *__restrict__ unitig_tip,
                            uint32_t *__restrict__ tip_reads) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const int32_t q = unitig_tip[step_unitig[t]];
    if (q >= 0) atomicAdd(&tip_reads[q], 1u);
}

// cs_a / ln_a > cs_b / ln_b, exactly: cs < 2^62 and ln < 2^31 (as branch_beats), so the products fit in 128 bits
__device__ __forceinline__ bool mean_above(const unsigned long long cs_a, const unsigned long long ln_a,
                                           const unsigned long long cs_b, const unsigned long long ln_b) {
    const unsigned long long lh = __umul64hi(cs_a, ln_b), rh = __umul64hi(cs_b, ln_a);
    if (lh != rh) return lh > rh;
    return cs_a * ln_b > cs_b * ln_a;
}

// one warp per tip: clip[q] = 1 when the tip has fewer than min_length nodes, is not spared, and an edge of
// list(attach) leads into another unitig whose mean node coverage is strictly larger.  The clipped tips are counted
// with one atomic per warp.
__global__ void k_tip_policy(const int32_t *__restrict__ tip_unitig, const int32_t *__restrict__ tip_attach, const long long Q,
                             const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges, const long long N,
                             const int32_t *__restrict__ e_tgt, const int32_t *__restrict__ node_unitig,
                             const int64_t *__restrict__ unitig_off, const unsigned long long *__restrict__ cov_sum,
                             const uint8_t *__restrict__ spared, const long long min_length, uint8_t *__restrict__ clip,
                             unsigned long long *__restrict__ n_clipped) {
    const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q >= Q) return;  // whole warps: Q is per warp
    const int32_t b = tip_unitig[q];
    const unsigned long long ln = (unsigned long long)(unitig_off[b + 1] - unitig_off[b]), cs = cov_sum[b];
    bool hit = false;
    if ((long long)ln < min_length && !spared[q]) {
        const int32_t a = tip_attach[q];
        const long long lo = adj_off[(a & 1) * N + (a >> 1)], hi = adj_off[(a & 1) * N + (a >> 1) + 1];
        for (long long i = lo + lane; i < hi && !hit; i += 32) {
            const int32_t c = node_unitig[e_tgt[adj_edges[i]]];
            hit = c != b && mean_above(cov_sum[c], (unsigned long long)(unitig_off[c + 1] - unitig_off[c]), cs, ln);
        }
    }
    const bool any = __any_sync(0xffffffffu, hit);
    if (lane == 0) {
        clip[q] = any ? 1 : 0;
        if (any) atomicAdd(n_clipped, 1ull);
    }
}

// one thread per read step on a clipped tip: an end clip (win >= 1, the step reaches the read's last window, window
// win - 1 live on state attach) drops the read's last `length` calls; a start clip (win == 0, the step is not the whole
// read, window `length` live on state attach ^ 1) drops its first `length` calls.  Dropped calls get code 1 in cnt.
__global__ void k_tip_clip(const int32_t *__restrict__ step_unitig, const int32_t *__restrict__ step_win,
                           const int32_t *__restrict__ step_length, const long long T, const int64_t *__restrict__ path_off,
                           const long long R, const int64_t *__restrict__ win_off, const int32_t *__restrict__ win_node,
                           const int8_t *__restrict__ win_dir, const int64_t *__restrict__ read_off,
                           const int32_t *__restrict__ unitig_tip, const int32_t *__restrict__ tip_attach,
                           const uint8_t *__restrict__ clip, uint32_t *__restrict__ cnt, uint8_t *__restrict__ changed,
                           uint32_t *__restrict__ clipped) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const int32_t q = unitig_tip[step_unitig[t]];
    if (q < 0 || !clip[q]) return;
    const long long r = segment_of(path_off, R, t);
    const long long w0 = win_off[r], nw = win_off[r + 1] - w0, i = step_win[t], l = step_length[t];
    const int32_t a = tip_attach[q];
    long long c0;
    if (i >= 1 && i + l == nw) {
        const int32_t n = win_node[w0 + i - 1];
        if (n < 0 || window_state(n, win_dir[w0 + i - 1]) != a) return;
        c0 = read_off[r + 1] - l;
    } else if (i == 0 && l < nw) {
        const int32_t n = win_node[w0 + l];
        if (n < 0 || window_state(n, win_dir[w0 + l]) != (a ^ 1)) return;
        c0 = read_off[r];
    } else {
        return;
    }
    for (long long j = 0; j < l; ++j) cnt[c0 + j] = 1u;
    changed[r] = 1;
    atomicAdd(&clipped[q], 1u);
}

}  // namespace amira
