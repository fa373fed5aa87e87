// stats.cuh -- the scans Amira runs right after a build, on the arrays the build left on the device
// (SURVEY.md 8f-1, 8f-4): reductions over the node -> reads CSR, the per-read lists and the adjacency CSR.
#pragma once

#include "post_kernels.cuh"

namespace amira {

constexpr int STAT_MAX_THRESHOLDS = 16;

struct Thresholds {
    int32_t min_len[STAT_MAX_THRESHOLDS];
    int n;
};

// get_overall_mean_node_coverages (graph_utils.py:299-313): for every threshold k, the number of
// (node, read) incidences whose read has at least k gene calls; the mean over nodes is sums[k] / N.
__global__ void k_read_length_coverages(const int64_t *__restrict__ reads_off, const uint32_t *__restrict__ reads,
                                        const int64_t *__restrict__ off, const long long n_inc, const int32_t read_base,
                                        const Thresholds T, unsigned long long *__restrict__ sums) {
    unsigned int cnt[STAT_MAX_THRESHOLDS];
#pragma unroll
    for (int t = 0; t < STAT_MAX_THRESHOLDS; ++t) cnt[t] = 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_inc; i += stride) {
        const long long r = (long long)reads[i] - read_base;
        const int len = (int)min((long long)0x7FFFFFFF, (long long)(off[r + 1] - off[r]));
#pragma unroll
        for (int t = 0; t < STAT_MAX_THRESHOLDS; ++t)
            if (t < T.n && len >= T.min_len[t]) ++cnt[t];
    }
#pragma unroll
    for (int t = 0; t < STAT_MAX_THRESHOLDS; ++t) {
        if (t >= T.n) break;
        unsigned int v = cnt[t];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&sums[t], (unsigned long long)v);
    }
}

// sum and maximum of the node coverages (get_all_node_coverages / get_mean_node_coverage, construct_graph.py:863-871)
__global__ void k_coverage_sum(const uint32_t *__restrict__ node_cov, const long long N, unsigned long long *__restrict__ out) {
    unsigned long long s = 0;
    unsigned int mx = 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
        const unsigned int c = node_cov[i];
        s += c;
        mx = max(mx, c);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, d);
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    }
    if ((threadIdx.x & 31) == 0) {
        if (s) atomicAdd(&out[0], s);
        if (mx) atomicMax(&out[1], (unsigned long long)mx);
    }
}

// remove_junk_reads (construct_graph.py:1398-1420): a read is rejected when more than
// round(n * (1 - error_rate)) of its n windows were filtered (None).  Python's round() on a float is
// round-half-to-even on the double product: rint() in the default rounding mode.
// mask: 0 = rejected, 1 = kept, 2 = short read (no entry in _readNodes).
__global__ void k_junk_read_mask(const int64_t *__restrict__ win_off, const int32_t *__restrict__ win_node,
                                 const uint8_t *__restrict__ is_short, const long long R, const double error_rate,
                                 uint8_t *__restrict__ mask) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    if (is_short[r]) {
        mask[r] = 2;
        return;
    }
    const long long a = win_off[r], b = win_off[r + 1];
    long long none = 0;
    for (long long w = a; w < b; ++w) none += win_node[w] < 0;
    const double expected = rint((double)(b - a) * (1.0 - error_rate));
    mask[r] = ((double)none <= expected) ? 1 : 0;
}

// get_nodes_containing (construct_graph.py:223-244): nodes whose canonical gene-mer holds one of the given
// genes (by rank, either strand)
__global__ void k_nodes_containing(const int32_t *__restrict__ node_key, const long long N, const int k,
                                   const int32_t *__restrict__ ranks, const int n_ranks, uint8_t *__restrict__ flags) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    bool hit = false;
    for (int j = 0; j < k && !hit; ++j) {
        const int g = abs(node_key[i * k + j]);
        for (int t = 0; t < n_ranks; ++t) hit |= g == ranks[t];
    }
    flags[i] = hit;
}

// remove_non_AMR_associated_nodes (construct_graph.py:2941-2959): reads of the flagged nodes, then the nodes
// that share no read with them
__global__ void k_mark_reads_of_nodes(const uint8_t *__restrict__ node_flag, const int64_t *__restrict__ reads_off,
                                      const uint32_t *__restrict__ reads, const long long N, const int32_t read_base,
                                      uint8_t *__restrict__ read_flag) {
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= N || !node_flag[warp]) return;
    for (long long i = reads_off[warp] + lane; i < reads_off[warp + 1]; i += 32) read_flag[(long long)reads[i] - read_base] = 1;
}

__global__ void k_nodes_with_marked_reads(const uint8_t *__restrict__ read_flag, const int64_t *__restrict__ reads_off,
                                          const uint32_t *__restrict__ reads, const long long N, const int32_t read_base,
                                          int *__restrict__ keep) {
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp > N) return;
    if (warp == N) {
        if (lane == 0) keep[N] = 0;
        return;
    }
    bool any = false;
    for (long long i = reads_off[warp] + lane; i < reads_off[warp + 1] && !any; i += 32) any = read_flag[(long long)reads[i] - read_base] != 0;
    any = __any_sync(0xffffffffu, any);
    if (lane == 0) keep[warp] = any;
}

// ---- linear chains (construct_graph.py:722-861) -------------------------------------------------------
// One step of upstream's path walk from a node: get_forward_node_from_node takes the forward edge only when it is
// the node's ONLY forward edge; get_backward_node_from_node takes the FIRST backward edge whenever there is one.
// Either way the walk extends when the target has degree 1 or 2 and is not the node itself.
// next = -1: no step; ext = walk continues; dir = direction in which the target is entered.
struct LinearSteps {
    int32_t *next[2];  // [0] forward, [1] backward
    int8_t *dir[2];
    uint8_t *ext[2];
    uint32_t *degree;
};

__device__ __forceinline__ void linear_step(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges,
                                            const int32_t *__restrict__ e_tgt, const int8_t *__restrict__ e_td, const long long N,
                                            const long long n, const int side, int32_t &nx, int8_t &d, uint8_t &ex) {
    const long long a0 = adj_off[side * N + n], a1 = adj_off[side * N + n + 1];
    const bool take = side ? (a1 > a0) : (a1 - a0 == 1);
    nx = -1;
    d = 0;
    ex = 0;
    if (take) {
        const uint32_t e = adj_edges[a0];
        nx = e_tgt[e];
        d = e_td[e];
        const long long deg = (adj_off[nx + 1] - adj_off[nx]) + (adj_off[N + nx + 1] - adj_off[N + nx]);
        ex = (deg == 1 || deg == 2) && nx != (int32_t)n;
    }
}

__global__ void k_linear_steps(const int64_t *__restrict__ adj_off, const uint32_t *__restrict__ adj_edges,
                               const int32_t *__restrict__ e_tgt, const int8_t *__restrict__ e_td, const long long N,
                               const LinearSteps S) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    S.degree[n] = (uint32_t)((adj_off[n + 1] - adj_off[n]) + (adj_off[N + n + 1] - adj_off[N + n]));
    for (int side = 0; side < 2; ++side) {
        int32_t nx;
        int8_t d;
        uint8_t ex;
        linear_step(adj_off, adj_edges, e_tgt, e_td, N, n, side, nx, d, ex);
        S.next[side][n] = nx;
        S.dir[side][n] = d;
        S.ext[side][n] = ex;
    }
}

}  // namespace amira
