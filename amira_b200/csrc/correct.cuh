// correct.cuh -- the reads through the simple bubbles rewritten along a kept branch (amira_gmg_correct_bubble_reads),
// over the cached read paths (unitigs.cuh) and bubbles (bubbles.cuh) and the build's input CSR.
//
// A read step on branch g (unitig b of m nodes, in bubble (sigma, tau)) is an edit when replace_with[g] >= 0, the
// step is m windows long, the windows win - 1 and win + m exist in its read and are live, and their states are
// (sigma, tau) (the read runs sigma -> b -> tau) or (tau ^ 1, sigma ^ 1) (the mirror).  The edit replaces the m calls
// [win, win + m) with the m' first genes of the kept branch's nodes, in the direction of travel.  Edits never overlap:
// every node of a branch has one-edge lists on both sides, and the junction nodes of a bubble have a list of two
// edges or more, so the flanking windows of an edit lie on no branch.
//
//  - k_correct_mark: one thread per read step tests the conditions (the step's read by binary search over path_off,
//    its bubble by binary search over branch_off).  An edit writes its signed m' (+: sigma -> tau) per step, and per
//    call a code: cnt = 0 untouched (one output call), 1 replaced and not the first (none), t + 2 the first replaced
//    call of the edit of step t (m' calls).  It flags its read and counts its branch with an integer atomic.
//  - one scan over the G calls turns the codes into every call's output index (idx[G] = the new call count).  The
//    reads are contiguous, so read r starts at idx[off[r]].
//  - k_correct_fill: one thread per call copies an untouched call and its positions; the thread of an edit's first
//    call writes the edit's m' genes.  k_correct_offsets writes the new read offsets.
#pragma once

#include "bubbles.cuh"

namespace amira {

// the segment of x in off[0..n] (off[0] <= x < off[n]): the last i with off[i] <= x
__device__ __forceinline__ long long segment_of(const int64_t *__restrict__ off, const long long n, const long long x) {
    long long lo = 0, hi = n;
    while (hi - lo > 1) {
        const long long mid = (lo + hi) >> 1;
        if (off[mid] <= x) lo = mid;
        else hi = mid;
    }
    return lo;
}

__global__ void k_correct_mark(const int32_t *__restrict__ step_unitig, const int32_t *__restrict__ step_win,
                               const int32_t *__restrict__ step_length, const long long T, const int64_t *__restrict__ path_off,
                               const long long R, const int64_t *__restrict__ win_off, const int32_t *__restrict__ win_node,
                               const int8_t *__restrict__ win_dir, const int64_t *__restrict__ read_off,
                               const int64_t *__restrict__ unitig_off, const int32_t *__restrict__ unitig_branch,
                               const int64_t *__restrict__ branch_off, const long long B, const int32_t *__restrict__ source,
                               const int32_t *__restrict__ sink, const int32_t *__restrict__ branch_unitig,
                               const int32_t *__restrict__ replace_with, uint32_t *__restrict__ cnt, int32_t *__restrict__ step_new,
                               uint8_t *__restrict__ changed, uint32_t *__restrict__ rewritten) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const int32_t b = step_unitig[t], g = unitig_branch[b];
    if (g < 0) return;
    const int32_t keep = replace_with[g];
    if (keep < 0) return;
    const long long m = unitig_off[b + 1] - unitig_off[b];
    if ((long long)step_length[t] != m) return;
    const long long r = segment_of(path_off, R, t);
    const long long w0 = win_off[r], nw = win_off[r + 1] - w0, i = step_win[t];
    if (i < 1 || i + m >= nw) return;
    const int32_t np = win_node[w0 + i - 1], nn = win_node[w0 + i + m];
    if (np < 0 || nn < 0) return;
    const int32_t sp = window_state(np, win_dir[w0 + i - 1]), sn = window_state(nn, win_dir[w0 + i + m]);
    const long long q = segment_of(branch_off, B, g);
    const int32_t sigma = source[q], tau = sink[q];
    const int dir = (sp == sigma && sn == tau) ? 1 : (sp == (tau ^ 1) && sn == (sigma ^ 1)) ? -1 : 0;
    if (dir == 0) return;
    const int32_t kb = branch_unitig[keep];
    const int32_t m2 = (int32_t)(unitig_off[kb + 1] - unitig_off[kb]);
    const long long c0 = read_off[r] + i;
    cnt[c0] = (uint32_t)(t + 2);
    for (long long j = 1; j < m; ++j) cnt[c0 + j] = 1u;
    step_new[t] = dir * m2;
    changed[r] = 1;
    atomicAdd(&rewritten[g], 1u);
}

struct CorrectCountLoad {
    const uint32_t *cnt;
    const int32_t *step_new;
    __device__ __forceinline__ unsigned long long operator()(long long c) const {
        const uint32_t v = cnt[c];
        return v == 0u ? 1ull : v == 1u ? 0ull : (unsigned long long)abs(step_new[v - 2u]);
    }
};
// ... -> idx[c] = the output index of call c; idx[G] = *n_out = the new call count
struct CorrectIndexStore {
    int64_t *idx;
    long long G;
    unsigned long long *n_out;
    __device__ __forceinline__ void operator()(long long c, unsigned long long excl, unsigned long long) const {
        idx[c] = (int64_t)excl;
        if (c == G) *n_out = excl;
    }
};

// out_* may be NULL (not asked for); ps / pe NULL without positions
__global__ void k_correct_fill(const uint32_t *__restrict__ cnt, const int64_t *__restrict__ idx, const long long G,
                               const int32_t *__restrict__ ids, const int32_t *__restrict__ ps, const int32_t *__restrict__ pe,
                               const int32_t *__restrict__ step_new, const int32_t *__restrict__ step_unitig,
                               const int32_t *__restrict__ step_length, const int32_t *__restrict__ unitig_branch,
                               const int32_t *__restrict__ replace_with, const int32_t *__restrict__ branch_unitig,
                               const int8_t *__restrict__ branch_orient, const int64_t *__restrict__ unitig_off,
                               const int32_t *__restrict__ unitig_nodes, const int8_t *__restrict__ node_orient,
                               const int32_t *__restrict__ key, const int k, int32_t *__restrict__ out_ids,
                               int32_t *__restrict__ out_ps, int32_t *__restrict__ out_pe) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= G) return;
    const uint32_t v = cnt[c];
    if (v == 1u) return;
    const long long o = idx[c];
    if (v == 0u) {
        if (out_ids) out_ids[o] = ids[c];
        if (out_ps && ps) out_ps[o] = ps[c];
        if (out_pe && pe) out_pe[o] = pe[c];
        return;
    }
    const long long t = (long long)v - 2;
    const int32_t s = step_new[t], m2 = abs(s);
    const int32_t keep = replace_with[unitig_branch[step_unitig[t]]];
    const int32_t kb = branch_unitig[keep];
    const int walk = (s > 0 ? 1 : -1) * branch_orient[keep];  // +1: the kept branch in its listed order
    const long long lo = unitig_off[kb], last = (long long)step_length[t] - 1;
    for (int32_t j = 0; j < m2; ++j) {
        if (out_ids) {
            const int32_t n = unitig_nodes[walk > 0 ? lo + j : lo + m2 - 1 - j];
            const int32_t *kn = key + (long long)n * k;
            out_ids[o + j] = walk * node_orient[n] > 0 ? kn[0] : -kn[k - 1];
        }
        const long long src = c + min((long long)j, last);
        if (out_ps && ps) out_ps[o + j] = ps[src];
        if (out_pe && pe) out_pe[o + j] = pe[src];
    }
}

__global__ void k_correct_offsets(const int64_t *__restrict__ read_off, const long long R, const int64_t *__restrict__ idx,
                                  int64_t *__restrict__ out_off) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r <= R) out_off[r] = idx[read_off[r]];
}

}  // namespace amira
