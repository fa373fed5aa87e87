// common.cuh -- error plumbing, device buffers, hashing and table slot layouts shared by the
// GeneMerGraph kernels.  sm_100a only.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <utility>

#include "../../include/amira_gmg.h"

namespace amira {

void set_error(const char *fmt, ...);

#define AMIRA_CUDA(expr)                                                                       \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            amira::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,              \
                             cudaGetErrorString(_e));                                          \
            return _e == cudaErrorMemoryAllocation ? AMIRA_E_NOMEM : AMIRA_E_CUDA;             \
        }                                                                                      \
    } while (0)

#define AMIRA_TRY(expr)                \
    do {                               \
        int _s = (expr);               \
        if (_s != AMIRA_OK) return _s; \
    } while (0)

// Bumped whenever a device buffer is reallocated or two buffers trade places.  Its one reader is the replay key of a
// captured build (GraphKey in gmg.cu): a captured CUDA graph holds raw pointers, so it may only be replayed while the
// generation it was captured at is still current.
inline std::atomic<uint64_t> &buffer_generation() {
    static std::atomic<uint64_t> g{0};
    return g;
}

// grow-only device allocation, reused across builds (Amira rebuilds the graph ~10-100x per sample).  The owner frees
// it; it must be destroyed while its device is current.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept { swap(o); }
    DevBuf &operator=(DevBuf &&o) noexcept {
        swap(o);
        o.release();
        return *this;
    }
    ~DevBuf() { release(); }
    int reserve(size_t bytes) {
        if (bytes <= cap) return AMIRA_OK;
        buffer_generation()++;
        release();
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            e = cudaMalloc(&p, bytes);
            want = bytes;
        }
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
            return AMIRA_E_NOMEM;
        }
        cap = want;
        return AMIRA_OK;
    }
    // two buffers trading places: a graph captured before holds the other one's pointer
    void swap(DevBuf &o) {
        std::swap(p, o.p);
        std::swap(cap, o.cap);
        buffer_generation()++;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T *as() const {
        return reinterpret_cast<T *>(p);
    }
};

// ---- table layouts -----------------------------------------------------------------------------
// Node table slot (32 B, one sector).  `word` packs, from the top: a 22-bit fingerprint
// of the canonical gene-mer, the 41-bit global call index p of the FIRST window seen with this
// gene-mer, and one bit that is set when that first window was the reverse complement of the
// canonical form.  Because the fingerprint is a function of the key, atomicMin over words of one
// key is atomicMin over p: the slot always names the first occurrence in (read, window) order,
// which is upstream's dict insertion order, and carries that occurrence's direction.
// The key itself is not stored: it is ids[p .. p+k) (reverse-complemented when the bit is set).
// `cov` counts from 0xFFFFFFFF so that the whole table is initialised by one memset(0xFF).
// klo / khi: the canonical gene-mer packed into up to 124 bits (when it fits), published by the thread
// that claimed the slot; all-ones = not (yet) published.
struct __align__(32) NodeSlot {
    unsigned long long word;
    unsigned int cov;  // occurrences - 1
    unsigned int aux;  // node index once the first-seen order is known
    unsigned long long klo, khi;
};
static_assert(sizeof(NodeSlot) == 32, "NodeSlot must be 32 bytes (one sector)");

constexpr unsigned long long EMPTY64 = ~0ull;
constexpr int P_BITS = 41;
constexpr unsigned long long P_MASK = (1ull << P_BITS) - 1;
constexpr int FP_SHIFT = P_BITS + 1;
constexpr unsigned int FP_MAX = (1u << (64 - FP_SHIFT)) - 2;  // all-ones is reserved for EMPTY

// Edge table slot (32 B = one sector).  One entry per UNDIRECTED adjacency {lo, hi, rel}: lo <= hi
// are node-table slot numbers, rel = sd*td.  Upstream creates two directed Edge objects per
// adjacent window pair (forward S->T and reverse T->S, construct_graph.py:246-262) whose identity
// is (source, target, sd*td) (construct_edge.py:104-124); both are always created by the same pair
// event and always have equal coverage, so one entry suffices: `ord` = (p << 2 | source_is_hi << 1
// | sd < 0) of the first pair event (atomicMin), from which both directed edges, their creation
// order (forward then reverse) and their stored directions follow.  S == T collapses to one
// directed edge with twice the count.
struct __align__(32) EdgeSlot {
    unsigned long long key;  // lo << 32 | hi << 1 | (rel > 0)
    unsigned long long ord;
    unsigned int cov;  // pair events - 1
    unsigned int pad[3];
};
static_assert(sizeof(EdgeSlot) == 32, "EdgeSlot must be 32 bytes");

// ---- compact layouts -----------------------------------------------------------------------------
// Random sector accesses are ~4x cheaper while the tables fit in L2 (measured: 1.9e11 RED/s and
// 2.8e11 sector loads/s into 64 MB, 4e10 and 9e10 into 170 MB), so the common case gets 16-byte slots:
//
// NodeSlot16: the canonical gene-mer itself (k genes x b bits <= 85 bits) is the identity: its top
// 22 bits sit where NodeSlot keeps the fingerprint (so word is still fingerprint | first position |
// first direction, and atomicMin over words of one gene-mer is atomicMin over positions), the low
// 63 bits are published in `key` by the thread that claimed the slot (all-ones = not yet published;
// a valid key has the top bit clear).  Coverage and node index live in side arrays.
struct __align__(16) NodeSlot16 {
    unsigned long long word;
    unsigned long long key;
};
// EdgeSlot16: as EdgeSlot with a 32-bit `ord` (call positions below 2^30).
struct __align__(16) EdgeSlot16 {
    unsigned long long key;
    unsigned int cov;  // pair events - 1
    unsigned int ord;
};
constexpr int KEY16_BITS = 85;       // 63 in NodeSlot16::key + 22 in the fingerprint field
constexpr int ORD32_P_BITS = 30;

// layout-independent view of the local node table for the passes after the insert
// info[slot] = {node index once the first-seen order is known, unit of that node's read list (incidence.cuh)}:
// one 8-byte gather per window in the partition pass
struct NodeView {
    unsigned long long *word;
    unsigned int *cov;
    uint2 *info;
    int wstride;  // in 64-bit words
    int cstride;  // in 32-bit words
    unsigned int cap;
    __device__ __forceinline__ unsigned long long w(unsigned int s) const { return word[(size_t)s * wstride]; }
    __device__ __forceinline__ unsigned int &c(unsigned int s) const { return cov[(size_t)s * cstride]; }
    __device__ __forceinline__ unsigned int &a(unsigned int s) const { return info[s].x; }
    __device__ __forceinline__ unsigned int &base(unsigned int s) const { return info[s].y; }
};

struct EdgeView {
    void *base;
    unsigned int cap;
    int compact;
    __device__ __forceinline__ bool get(unsigned int s, unsigned long long &key, unsigned long long &ord,
                                        unsigned int &cov) const {
        if (compact) {
            const EdgeSlot16 e = reinterpret_cast<const EdgeSlot16 *>(base)[s];
            key = e.key;
            ord = e.ord;
            cov = e.cov;
        } else {
            const EdgeSlot *e = reinterpret_cast<const EdgeSlot *>(base) + s;
            key = e->key;
            ord = e->ord;
            cov = e->cov;
        }
        return key != ~0ull;
    }
};

// ---- multi-GPU plumbing (comm.cu) ----------------------------------------------------------------
struct Comm;
int comm_unique_id(void *out_128_bytes);
int comm_create(Comm **out, const void *unique_id, int rank, int world);
void comm_destroy(Comm *c);
int comm_rank(const Comm *c);
int comm_world(const Comm *c);
int comm_allgather(Comm *c, const void *d_send, void *d_recv, size_t bytes_per_rank, cudaStream_t st);
int comm_allreduce_max_i32(Comm *c, int *d_buf, int n, cudaStream_t st);
int comm_alltoallv(Comm *c, const void *d_send, const int64_t *send_off, void *d_recv, const int64_t *recv_off,
                   size_t elem_bytes, cudaStream_t st);
int comm_allgatherv(Comm *c, const void *d_send, int64_t n_send, void *d_recv, const int64_t *recv_off,
                    size_t elem_bytes, cudaStream_t st);
int comm_window_ensure(Comm *c, size_t need_bytes, cudaStream_t st);  // collective; same need_bytes on every rank
bool comm_p2p(const Comm *c);
void *comm_window(const Comm *c, int p);
int comm_barrier(Comm *c, cudaStream_t st);

// L2 eviction-priority hints: the small, randomly revisited arrays (hash tables, slot info, the write frontier
// of the raw read lists) are kept with evict_last while the window arrays stream past with evict_first loads
__device__ __forceinline__ unsigned long long l2_evict_last_policy() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void st_u32_hint(uint32_t *p, uint32_t v, unsigned long long pol) {
    asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ uint2 ld_u32x2_hint(const uint2 *p, unsigned long long pol) {
    uint2 v;
    asm volatile("ld.global.L2::cache_hint.v2.u32 {%0, %1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
    return v;
}

__host__ __device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return x;
}

}  // namespace amira
