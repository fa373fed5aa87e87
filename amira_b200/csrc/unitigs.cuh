// unitigs.cuh -- the compacted graph (SURVEY.md 8f-4): every maximal non-branching path of the gene-mer graph as one
// unitig, by list ranking over the 2N states of the adjacency CSR.
//
// A state is s = 2 * node + side (side 0 = leaving through the forward list, 1 = through the backward list).
// succ(2u + a) = 2v + (td == 1 ? 0 : 1) when list a of u holds exactly one edge e = (u -> v, td), v != u, and v's
// entering list (backward when td = +1, forward when td = -1: where the reverse of e lives) holds exactly one edge.
// The rule is symmetric: succ(s) = t <=> succ(t ^ 1) = s ^ 1 (the reverse of the one edge of s is the one edge of
// t ^ 1, and both lists hold one edge).  So every state has at most one successor and one predecessor, and the
// states form disjoint simple paths and cycles.  A chain never holds both states of one node: its middle would need a
// step with v = u.  Self edges of either sign are excluded by v != u; multi-edges between two nodes put two edges in
// one list of one of them (condition 1 or 3 fails).  A chain and its mirror (every state ^ 1) are one unitig.
//
//  - ranking: Wyllie over ping-pong (pointer, distance, running minimum) arrays, ceil(log2 S) + 1 rounds: every path
//    state ends at its tail with its distance to it and the minimum state from it to the tail; every cycle state
//    ends with the minimum of its whole cycle (2^rounds > S steps covered).
//  - cycles: a state whose pointer does not end at a terminal lies on a cycle; the cycle's minimum state is cut
//    (made a terminal) and the distances are ranked again, only when a cycle exists.
//  - per node n: the chain minimum of 2n is min(mn[2n], mn[2n + 1] ^ 1) (a mirror segment holds one state per node,
//    so its minimum is the mirror of the segment's minimum); the unitig is listed in the orientation whose chain
//    holds the even state 2m of its smallest node m, so n is listed through 2n when that minimum is even, through
//    2n + 1 otherwise.  Its position from the head is dist[s ^ 1]: on a path the mirror runs from s ^ 1 to the
//    mirror of the head; on a cycle the mirror is cut at 2m + 1, so it runs from s ^ 1 back to the mirror of m.
//  - numbering: a scan over the nodes flagged "n is its unitig's m" gives the ids, a scan over the unitig lengths
//    the offsets; every node scatters itself to unitig_nodes[off[id] + pos] (a permutation: no atomics), its
//    coverage to the unitig's sum / min / max (atomics per unitig).
//  - edges: a directed edge of list a of node u joins consecutive nodes of one unitig iff succ(2u + a) exists.
// The jump table of paths.cuh (S x L x 4 bytes) is not needed here: memory is 7 x S x 4 bytes for the ranking plus
// O(N + E) for the results.  The cycle kernels of paths.cuh work on that table's levels and do not apply.
//
// The edges and the reads of the compacted graph, over the cached succ / node_unitig / node_pos / node_orient:
//  - links: a scan over the directed edges flagged "edge_internal == 0" compacts the junction edges in edge order;
//    one thread per link (k_unitig_links) then writes its unitig ends: from (node_unitig[u], sd * node_orient[u])
//    to (node_unitig[v], td * node_orient[v]), and the edge's coverage.
//  - read paths: a window on node n with direction d leaves n through the state 2n + (d < 0), as the edge the
//    build made from it and the next window does.  A window continues the window before it when both are live
//    (not None), in one read, and succ(state of the one before) == its state.  One thread per window
//    (k_read_step_flags) flags "starts a step" (live, does not continue) and "ends a step" (live, the next window
//    does not continue it); one scan over the W windows numbers the steps and, at a start, writes the step's
//    unitig, orientation, position and window index, at an end the step's last window + 1; at each read's first
//    window it writes path_off (also for the short reads before it, which have no windows).  A None window starts
//    and ends nothing, so a step's length comes from its own end, not from the next step's start:
//    k_read_step_lengths subtracts.  Window and step numbers are 64-bit; a window's index within its read and a
//    step's length are 32-bit.
#pragma once

#include "stats.cuh"

namespace amira {

// number of edges in list `side` (0 = forward, 1 = backward) of node n
__device__ __forceinline__ long long adj_list_size(const int64_t *__restrict__ adj_off, const long long N, const long long n,
                                                   const int side) {
    return adj_off[side * N + n + 1] - adj_off[side * N + n];
}

__device__ __forceinline__ int32_t unitig_step(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges,
                                               const int32_t *__restrict__ e_tgt, const int8_t *__restrict__ e_td,
                                               const long long N, const long long u, const int side) {
    if (adj_list_size(adj_off, N, u, side) != 1) return -1;
    const uint32_t e = adj_edges[adj_off[side * N + u]];
    const int32_t v = e_tgt[e];
    const int leave = e_td[e] == 1 ? 0 : 1;
    if (v == (int32_t)u || adj_list_size(adj_off, N, v, leave ^ 1) != 1) return -1;
    return 2 * v + leave;
}

// succ, and round 0 of the ranking: ptr = succ (itself at a terminal), dist = steps taken, mn = the state itself
__global__ void k_unitig_succ(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges,
                              const int32_t *__restrict__ e_tgt, const int8_t *__restrict__ e_td, const long long N,
                              int32_t *__restrict__ succ, int32_t *__restrict__ ptr, uint32_t *__restrict__ dist,
                              int32_t *__restrict__ mn) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= 2 * N) return;
    const int32_t t = unitig_step(adj_off, adj_edges, e_tgt, e_td, N, s >> 1, (int)(s & 1));
    succ[s] = t;
    ptr[s] = t < 0 ? (int32_t)s : t;
    dist[s] = t < 0 ? 0u : 1u;
    mn[s] = (int32_t)s;
}

// one Wyllie round; mn_in == nullptr: distances only.  Distances saturate at S (they only grow without bound around a
// cycle, where they are not used)
__global__ void k_unitig_rank_round(const int32_t *__restrict__ p_in, const uint32_t *__restrict__ d_in,
                                    const int32_t *__restrict__ m_in, int32_t *__restrict__ p_out, uint32_t *__restrict__ d_out,
                                    int32_t *__restrict__ m_out, const long long S) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int32_t p = p_in[s];
    p_out[s] = p_in[p];
    d_out[s] = (uint32_t)min((unsigned long long)d_in[s] + d_in[p], (unsigned long long)S);
    if (m_in) m_out[s] = min(m_in[s], m_in[p]);
}

// after the first ranking: circ[n] = node n lies on a cycle; the cycles are cut at their minimum state and round 0
// of the second ranking is written to (p_out, d_out); *any_cycle = 1 when there is a cycle
__global__ void k_unitig_cycle_cut(const int32_t *__restrict__ succ, const int32_t *__restrict__ ptr, const int32_t *__restrict__ mn,
                                   int32_t *__restrict__ p_out, uint32_t *__restrict__ d_out, uint8_t *__restrict__ circ,
                                   int *__restrict__ any_cycle, const long long S) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int32_t t = succ[s];
    const bool cyc = succ[ptr[s]] >= 0;
    const bool cut = t < 0 || (cyc && mn[s] == (int32_t)s);
    p_out[s] = cut ? (int32_t)s : t;
    d_out[s] = cut ? 0u : 1u;
    if ((s & 1) == 0) circ[s >> 1] = cyc ? 1 : 0;
    if (cyc && mn[s] == (int32_t)s) *any_cycle = 1;
}

struct UnitigRanks {
    const int32_t *succ, *mn;
    const uint32_t *dist;   // final distances (cycles cut at their minimum state)
    const uint8_t *circ;
    // the state node n is listed through, and its unitig's smallest node
    __device__ __forceinline__ int32_t listed(long long n, int32_t &m) const {
        const int32_t cm = min(mn[2 * n], mn[2 * n + 1] ^ 1);
        m = cm >> 1;
        return (int32_t)(2 * n + (cm & 1));
    }
};

// scan 1 over the nodes: 1 where n is its unitig's smallest node
struct UnitigHeadLoad {
    UnitigRanks R;
    __device__ __forceinline__ unsigned long long operator()(long long n) const {
        int32_t m;
        R.listed(n, m);
        return m == (int32_t)n ? 1ull : 0ull;
    }
};
// ... -> uid[n] = ids of the heads; per unitig its length and circular flag, coverage accumulators cleared;
// *n_unitigs = U
struct UnitigHeadStore {
    UnitigRanks R;
    int32_t *uid;
    uint32_t *len;
    uint8_t *circular;
    unsigned long long *cov_sum;
    uint32_t *cov_min, *cov_max;
    long long N;
    long long *n_unitigs;
    __device__ __forceinline__ void operator()(long long n, unsigned long long excl, unsigned long long head) const {
        if (n == N) {
            *n_unitigs = (long long)excl;
            return;
        }
        uid[n] = (int32_t)excl;
        if (!head) return;
        const bool c = R.circ[n];
        // listed through 2n: a path's length is both distances + 1, a cycle's the distance of succ(2n) to 2n + 1
        len[excl] = c ? R.dist[R.succ[2 * n]] + 1 : R.dist[2 * n] + R.dist[2 * n + 1] + 1;
        circular[excl] = c ? 1 : 0;
        cov_sum[excl] = 0;
        cov_min[excl] = 0xFFFFFFFFu;
        cov_max[excl] = 0;
    }
};

// scan 2 over the unitigs: their offsets into unitig_nodes
struct UnitigLenLoad {
    const uint32_t *len;
    __device__ __forceinline__ unsigned long long operator()(long long u) const { return len[u]; }
};
struct UnitigOffStore {
    int64_t *off;
    __device__ __forceinline__ void operator()(long long u, unsigned long long excl, unsigned long long) const { off[u] = (int64_t)excl; }
};

__global__ void k_unitig_scatter(const UnitigRanks R, const int32_t *__restrict__ uid, const int64_t *__restrict__ off,
                                 const uint32_t *__restrict__ node_cov, const long long N, int32_t *__restrict__ node_unitig,
                                 int32_t *__restrict__ node_pos, int8_t *__restrict__ node_orient, int32_t *__restrict__ unitig_nodes,
                                 unsigned long long *__restrict__ cov_sum, uint32_t *__restrict__ cov_min,
                                 uint32_t *__restrict__ cov_max) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    int32_t m;
    const int32_t s = R.listed(n, m);
    const int32_t id = uid[m];
    const int32_t pos = (int32_t)R.dist[s ^ 1];
    node_unitig[n] = id;
    node_pos[n] = pos;
    node_orient[n] = (s & 1) ? -1 : 1;
    unitig_nodes[off[id] + pos] = (int32_t)n;
    const uint32_t c = node_cov[n];
    atomicAdd(&cov_sum[id], (unsigned long long)c);
    atomicMin(&cov_min[id], c);
    atomicMax(&cov_max[id], c);
}

__global__ void k_unitig_edges(const int32_t *__restrict__ succ, const int32_t *__restrict__ e_src, const int8_t *__restrict__ e_sd,
                               const long long E, uint8_t *__restrict__ internal) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= E) return;
    internal[j] = succ[2 * (long long)e_src[j] + (e_sd[j] < 0 ? 1 : 0)] >= 0 ? 1 : 0;
}

// ---- links: the junction edges, in edge order --------------------------------------------------------------------
struct JunctionLoad {
    const uint8_t *internal;
    __device__ __forceinline__ unsigned long long operator()(long long j) const { return internal[j] ? 0ull : 1ull; }
};
// ... -> link_edge[excl] = j for a junction; *n_links = L
struct JunctionStore {
    int32_t *link_edge;
    long long E;
    long long *n_links;
    __device__ __forceinline__ void operator()(long long j, unsigned long long excl, unsigned long long junction) const {
        if (j == E) *n_links = (long long)excl;
        else if (junction) link_edge[excl] = (int32_t)j;
    }
};

__global__ void k_unitig_links(const int32_t *__restrict__ link_edge, const long long L, const int32_t *__restrict__ e_src,
                               const int32_t *__restrict__ e_tgt, const int8_t *__restrict__ e_sd, const int8_t *__restrict__ e_td,
                               const uint32_t *__restrict__ e_cov, const int32_t *__restrict__ node_unitig,
                               const int8_t *__restrict__ node_orient, int32_t *__restrict__ from_unitig,
                               int8_t *__restrict__ from_orient, int32_t *__restrict__ to_unitig, int8_t *__restrict__ to_orient,
                               uint32_t *__restrict__ cov) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= L) return;
    const int32_t j = link_edge[t], u = e_src[j], v = e_tgt[j];
    from_unitig[t] = node_unitig[u];
    from_orient[t] = (int8_t)(e_sd[j] * node_orient[u]);
    to_unitig[t] = node_unitig[v];
    to_orient[t] = (int8_t)(e_td[j] * node_orient[v]);
    cov[t] = e_cov[j];
}

// ---- read paths: maximal runs of windows that follow succ ---------------------------------------------------------
constexpr uint8_t STEP_START = 1, STEP_END = 2;

// the state a live window leaves its node through
__device__ __forceinline__ int32_t window_state(const int32_t n, const int8_t d) { return 2 * n + (d < 0 ? 1 : 0); }

__global__ void k_read_step_flags(const int32_t *__restrict__ win_node, const int8_t *__restrict__ win_dir,
                                  const int32_t *__restrict__ win_read, const long long W, const int32_t *__restrict__ succ,
                                  uint8_t *__restrict__ flags) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    const int32_t n = win_node[w];
    if (n < 0) {
        flags[w] = 0;
        return;
    }
    const int32_t s = window_state(n, win_dir[w]), r = win_read[w];
    bool in = false, out = false;  // w continues w - 1; w + 1 continues w
    if (w > 0 && win_read[w - 1] == r) {
        const int32_t p = win_node[w - 1];
        in = p >= 0 && succ[window_state(p, win_dir[w - 1])] == s;
    }
    if (w + 1 < W && win_read[w + 1] == r) {
        const int32_t q = win_node[w + 1];
        out = q >= 0 && succ[s] == window_state(q, win_dir[w + 1]);
    }
    flags[w] = (in ? 0 : STEP_START) | (out ? 0 : STEP_END);
}

struct StepLoad {
    const uint8_t *flags;
    __device__ __forceinline__ unsigned long long operator()(long long w) const { return flags[w] & STEP_START; }
};
// ... -> path_off of the reads whose windows begin at w; at a start the step's fields (length = the end of the step
// within its read, until k_read_step_lengths); *n_steps = T
struct StepStore {
    const uint8_t *flags;
    const int32_t *win_node, *win_read;
    const int8_t *win_dir;
    const int64_t *win_off;
    const int32_t *node_unitig, *node_pos;
    const int8_t *node_orient;
    long long W, R;
    int64_t *path_off;
    int32_t *unitig, *pos, *win, *length;
    int8_t *orient;
    long long *n_steps;
    __device__ __forceinline__ void operator()(long long w, unsigned long long excl, unsigned long long start) const {
        const long long r = w < W ? (long long)win_read[w] : R;
        for (long long q = w > 0 ? (long long)win_read[w - 1] + 1 : 0; q <= r; ++q) path_off[q] = (int64_t)excl;
        if (w == W) {
            *n_steps = (long long)excl;
            return;
        }
        const uint8_t f = flags[w];
        if (!f) return;
        const long long first = win_off[r];
        if (start) {
            const int32_t n = win_node[w];
            unitig[excl] = node_unitig[n];
            orient[excl] = (int8_t)((win_dir[w] < 0 ? -1 : 1) * node_orient[n]);
            pos[excl] = node_pos[n];
            win[excl] = (int32_t)(w - first);
        }
        if (f & STEP_END) length[excl + start - 1] = (int32_t)(w + 1 - first);
    }
};

__global__ void k_read_step_lengths(const int32_t *__restrict__ win, const long long T, int32_t *__restrict__ length) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < T) length[t] -= win[t];
}

}  // namespace amira
