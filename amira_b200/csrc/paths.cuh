// paths.cuh -- linear walks (get_forward_path_from_node / get_backward_path_from_node, construct_graph.py:722-848)
// from many start points at once, by pointer jumping over the 2N walk states (SURVEY.md 8f-4).
//
// A state is s = 2 * node + side (side 0 = forward list, 1 = backward list).  One step of upstream's walk
// (linear_step, stats.cuh) gives succ(s) = 2 * next + (dir == 1 ? 0 : 1) when the walk extends, none otherwise.
// succ is a functional graph: every state either runs into a terminal (a state without successor) or into a cycle.
//  - jump table: J[l][s] = succ^(2^l)(s), -1 once a terminal is passed; L levels with 2^L > 2N, so every walk
//    length and every cycle length is one O(L) descent.
//  - cycles: min-propagation over the table labels each cycle with its smallest state; cutting every cycle there
//    leaves a forest, ranked by pointer jumping: root[s] = the terminal or cycle label s runs into, dist[s] = steps.
//  - a query s0 (node n0) walks until a terminal or until the next state belongs to n0: the first hit of s0 ^ 1 or
//    of s0 itself follows from root / dist and one or two jumps, the cycle length from dist[succ(label)].
// Table: 2N * L * 4 bytes (170 MB at N = 10^6); everything else O(N + queries + output).
#pragma once

#include "stats.cuh"

namespace amira {

constexpr int32_t WALK_NEVER_ENDS = 0x7FFFFFFF;

// J[0] = succ, nxt = next node of the state (-1 none: also the node a want_branched walk appends)
__global__ void k_walk_succ(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges,
                            const int32_t *__restrict__ e_tgt, const int8_t *__restrict__ e_td, const long long N,
                            int32_t *__restrict__ succ, int32_t *__restrict__ nxt) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= 2 * N) return;
    int32_t nx;
    int8_t d;
    uint8_t ex;
    linear_step(adj_off, adj_edges, e_tgt, e_td, N, s >> 1, (int)(s & 1), nx, d, ex);
    succ[s] = ex ? 2 * nx + (d == 1 ? 0 : 1) : -1;
    nxt[s] = nx;
}

__global__ void k_walk_jump_level(const int32_t *__restrict__ prev, int32_t *__restrict__ cur, const long long S) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int32_t t = prev[s];
    cur[s] = t < 0 ? -1 : prev[t];
}

// m_out[s] = min over the 2^(l+1) states from s on, given m_in over 2^l (m_in == nullptr: the states themselves)
__global__ void k_walk_cycle_min(const int32_t *__restrict__ J_l, const int32_t *__restrict__ m_in, int32_t *__restrict__ m_out,
                                 const long long S) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int32_t t = J_l[s];
    const int32_t a = m_in ? m_in[s] : (int32_t)s;
    m_out[s] = t < 0 ? a : min(a, m_in ? m_in[t] : t);
}

// a state without terminal is 2^L > 2N steps from a state e on its cycle; the window min at e covers the whole cycle
__global__ void k_walk_cycle_labels(const int32_t *__restrict__ J_top, const int32_t *__restrict__ m, uint8_t *__restrict__ is_label,
                                    const long long S) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int32_t h = J_top[s];
    const int32_t e = h < 0 ? -1 : J_top[h];
    if (e >= 0) is_label[m[e]] = 1;
}

// forest with every cycle cut at its label: parent = succ, or the state itself at a terminal / label
__global__ void k_walk_rank_init(const int32_t *__restrict__ succ, const uint8_t *__restrict__ is_label, int32_t *__restrict__ root,
                                 int32_t *__restrict__ dist, const long long S) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int32_t t = succ[s];
    const bool cut = t < 0 || is_label[s];
    root[s] = cut ? (int32_t)s : t;
    dist[s] = cut ? 0 : 1;
}

__global__ void k_walk_rank_round(const int32_t *__restrict__ r_in, const int32_t *__restrict__ d_in, int32_t *__restrict__ r_out,
                                  int32_t *__restrict__ d_out, const long long S) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int32_t r = r_in[s];
    r_out[s] = r_in[r];
    d_out[s] = d_in[s] + d_in[r];
}

struct WalkTable {
    const int32_t *J;     // L levels of S states
    const int32_t *nxt, *root, *dist;
    long long S;
    int L;
    // succ^k(s) for 0 <= k < 2^L; -1 when the walk from s has fewer than k steps
    __device__ __forceinline__ int32_t jump(int32_t s, long long k) const {
        for (int l = 0; k && s >= 0; ++l, k >>= 1)
            if (k & 1) s = J[(long long)l * S + s];
        return s;
    }
    __device__ __forceinline__ bool on_cycle(int32_t s, long long clen) const { return jump(s, clen) == s; }
};

// steps[i] = number of steps of the walk from states[i] (WALK_NEVER_ENDS: it never ends, *bad = first such query);
// len[i] = nodes it outputs (plus the branching node)
__global__ void k_walk_lengths(const WalkTable T, const int32_t *__restrict__ states, const long long n, const int want_branched,
                               int32_t *__restrict__ steps, unsigned long long *__restrict__ len, int *__restrict__ bad) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t s0 = states[i], a = s0 ^ 1;
    const int32_t r = T.root[s0], ra = T.root[a];
    const long long d0 = T.dist[s0], da = T.dist[a];
    const int32_t succ_r = T.J[r];  // level 0
    long long k = -1;               // steps to the first state of n0 after s0 (-1: never)
    if (ra == r && da < d0 && T.jump(s0, d0 - da) == a) k = d0 - da;
    long long j;
    if (succ_r < 0) {
        j = k >= 0 ? k - 1 : d0;    // r is a terminal: the walk stops there unless it meets n0 first
    } else {
        const long long clen = (long long)T.dist[succ_r] + 1;  // r is the label of the cycle the walk runs around
        if (k < 0 && ra == r && T.on_cycle(a, clen)) k = d0 + clen - da;
        if (T.on_cycle(s0, clen)) k = k < 0 ? clen : min(k, clen);
        j = k >= 0 ? k - 1 : -1;
    }
    if (j < 0) {
        atomicMin(bad, (int)min(i, (long long)WALK_NEVER_ENDS - 1));
        steps[i] = WALK_NEVER_ENDS;
        len[i] = 0;
        return;
    }
    steps[i] = (int32_t)j;
    len[i] = (unsigned long long)j + (want_branched && T.nxt[T.jump(s0, j)] >= 0 ? 1 : 0);
}

struct WalkLenLoad {
    const unsigned long long *len;
    __device__ __forceinline__ unsigned long long operator()(long long i) const { return len[i]; }
};
struct WalkOffStore {
    int64_t *off;
    __device__ __forceinline__ void operator()(long long i, unsigned long long excl, unsigned long long) const { off[i] = (int64_t)excl; }
};

// one thread per output node: its query by binary search over the offsets, its node by one jump
__global__ void k_walk_fill(const WalkTable T, const int32_t *__restrict__ states, const long long n, const int64_t *__restrict__ off,
                            const int32_t *__restrict__ steps, int32_t *__restrict__ out) {
    const long long total = off[n];
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        long long lo = 0, hi = n - 1;  // last query with off[q] <= e
        while (lo < hi) {
            const long long mid = (lo + hi + 1) >> 1;
            if (off[mid] <= e) lo = mid;
            else hi = mid - 1;
        }
        const long long p = e - off[lo] + 1;
        const int32_t j = steps[lo];
        out[e] = p <= j ? T.jump(states[lo], p) >> 1 : T.nxt[T.jump(states[lo], j)];
    }
}

}  // namespace amira
