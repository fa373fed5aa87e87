// gmg.cu -- the handle, the build / filter pipelines and the C ABI of libamira_gmg.so.
// See include/amira_gmg.h for the contract, gmg_kernels.cuh for the insert kernel and
// post_kernels.cuh for the passes after it.
#include <stdarg.h>

#include <algorithm>
#include <vector>

#include "post_kernels.cuh"
#include "stats.cuh"
#include "sharded.cuh"

namespace amira {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

}  // namespace amira

using namespace amira;

struct amira_gmg {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    // Second stream: after the node order is known, (edges -> adjacency -> components) runs beside
    // (per-read lists -> node/read incidence); `cur` is what the launch helpers use.
    cudaStream_t stream2 = nullptr, cur = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // Third stream: the per-read exports are copied out as soon as the per-read lists are final
    // (ev_reads_ready: after the scatter pass of a build, after the masking of a filter), i.e. while the
    // incidence / adjacency / component passes of the same build are still running.
    cudaStream_t stream_copy = nullptr;
    cudaEvent_t ev_reads_ready = nullptr;
    // host input: the gene ids arrive in H2D_PIECES pieces on the copy stream; the insert kernel is
    // launched once per piece, as soon as the piece after it (its halo) has landed
    static constexpr int H2D_PIECES = 4;
    cudaEvent_t ev_h2d[H2D_PIECES] = {};
    cudaEvent_t ev_input_free = nullptr;
    int64_t piece_end[H2D_PIECES] = {};  // call index where each piece ends; 0 pieces = input already resident
    int n_pieces = 0;
    int n_sm = 148;
    int insert_ctas_per_sm = 1;
    int force_layout = 0;        // test hook (amira_gmg_debug_layout): 1 = no 16-byte node slots, 2 = no 16-byte edge slots, 4 = no packed keys, 8 = the 16384-bucket shape of the partition pass, 16 = units share buckets pairwise
    int id_bits = 0;             // bits a signed gene id takes in a packed key (from the largest |id| seen); 0 = unknown
    bool n16 = false, e16 = false;  // 16-byte node / edge slots in the current build
    NodeView nview;
    EdgeView eview;
    DevBuf d_maxabs;

    // input (owned copy or borrowed device pointers)
    DevBuf d_ids, d_off, d_ps, d_pe;
    const int32_t *ids = nullptr;
    const int64_t *off = nullptr;
    const int32_t *ps = nullptr, *pe = nullptr;
    int64_t R = 0, G = 0;
    int k = 0;
    bool has_pos = false;
    bool input_on_device = false;
    // device-resident input: the call count read_off[R] of the last build, reused while the same offsets
    // array is passed again (the per-read kernel verifies it on the device: ST_STALE)
    const int64_t *cache_off = nullptr;
    int64_t cache_R = -1, cache_G = 0;

    // per read / per tile
    DevBuf win_off, is_short, to_correct, tile_r0;
    // per window
    DevBuf win_slot, win_node, win_dir, win_read, win_start, win_end;  // win_slot: table slots from the insert kernel; win_node: node indices
    // node -> reads transpose (incidence.cuh): (node, read) records dealt into buckets, first node of every unit
    DevBuf inc_rec, unit_lo, bucket_cursor;
    UnitPlan unit_plan = {};
    // hash tables + first-seen bitmaps
    DevBuf ntab, etab, slot_info, bitmaps, cnt_node, cnt_edge;
    unsigned int ncap = 0, ecap = 0;
    int key_bits = 0;
    int64_t grow_n = 1, grow_e = 1;     // capacity multipliers after an overflow
    int64_t hint_nodes = 0, hint_edges = 0;
    int64_t filt_N = -1, filt_E = -1;  // node / edge counts before the last filter (keep flags are retained)
    int64_t prev_G = 0, prev_nodes = 0, prev_und_edges = 0;  // sizes of the previous build on this handle
    int64_t cap_nodes = 0, cap_edges = 0;  // capacities of the node / edge arrays of the current build
    // nodes (cur) and compaction targets (alt)
    DevBuf node_key, node_cov, node_dir, node_comp, reads_off, reads;
    DevBuf node_key2, node_cov2, node_dir2, node_comp2, reads_off2, reads2;
    DevBuf parent, is_root, cc_min, link, run_id, run_pairs;  // link: node i is joined to node i - 1; run_id: run of linked nodes
    // edges
    DevBuf e_src, e_tgt, e_sd, e_td, e_cov;
    DevBuf e_src2, e_tgt2, e_sd2, e_td2, e_cov2;
    // adjacency: adj_off[2N+1] (forward lists of all nodes, then backward lists), adj_edges[E]
    DevBuf adj_off, adj_edges, adj_cursor, adj_tmp, reads_tmp;
    // scratch
    DevBuf dups, seg_work[2], scan_state[2], keep_n, keep_e, comp_max, scratch_off;
    // tile states of all the scans of one build: cleared by ONE memset when the build is enqueued, handed out in pieces
    DevBuf scan_pool;
    size_t scan_pool_used = 0, scan_pool_ready = 0;
    DevBuf d_status, d_sizes;
    int *h_status = nullptr;       // pinned: [0] early copy, [ST_COUNT] final copy
    long long *h_sizes = nullptr;  // pinned: [0] early copy, [SZ_COUNT] final copy
    cudaEvent_t ev_early = nullptr, ev_done = nullptr;

    int64_t n_nodes = 0, n_edges = 0, W = 0, n_inc = 0, n_short = 0, n_fw = 0, n_bw = 0, n_comps = 0;
    bool built = false;
    // a build / filter has been enqueued and its status and sizes have not been looked at yet:
    // 0 = nothing pending, 1 = early sizes (nodes, edges, windows) taken, 2 = everything still pending
    int pending = 0;
    bool pending_is_build = false;
    int attempts = 0;
    int last_status = AMIRA_OK;

    // A build whose input pointers, sizes and table capacities repeat (the k sweep / rebuild loop over a resident
    // CSR, the small-graph regime where ~50 launches cost more than the kernels) is captured into a CUDA graph the
    // second time it is seen and replayed from then on.
    struct GraphKey {
        const void *ids, *off, *ps, *pe;
        int64_t R, G, cap_nodes, cap_edges;
        unsigned int ncap, ecap;
        int k, key_bits, layout;
        uint64_t buffers;  // buffer_generation() (common.cuh): the device buffers the graph was captured with
        bool operator==(const GraphKey &o) const {
            return ids == o.ids && off == o.off && ps == o.ps && pe == o.pe && R == o.R && G == o.G && cap_nodes == o.cap_nodes &&
                   cap_edges == o.cap_edges && ncap == o.ncap && ecap == o.ecap && k == o.k && key_bits == o.key_bits && layout == o.layout &&
                   buffers == o.buffers;
        }
    };
    GraphKey graph_key = {}, last_key = {};
    cudaGraphExec_t graph_exec = nullptr;
    bool capturing = false;
    int64_t graph_launches = 0, graph_kernels = 0;  // replays; kernels inside the captured graph

    bool profiling = false;
    cudaEvent_t ev[AMIRA_PH_COUNT][2] = {};
    bool ev_used[AMIRA_PH_COUNT] = {};
    int64_t launches = 0;      // hand-written kernels launched
    int64_t lib_launches = 0;  // memset / memcpy calls

    // multi-GPU (sharded.cuh): exchange scratch, local coverage per global node
    Comm *comm = nullptr;
    int rank = 0, world = 1;
    int64_t first_read_global = 0, first_call_global = 0, calls_global = 0;
    int64_t sh_Eg = 0;               // merged undirected edge records of the current sharded build
    const EdgeSlot *sh_gedge = nullptr;
    BuildParams local_P;             // parameters of the last k_insert_windows launch (the local tables)
    DevBuf x_cnt, x_skey, x_smeta, x_rkey, x_rmeta, x_rmeta2, x_mkey, x_mmeta, x_gkey, x_gmeta, x_tab,
        x_bm, x_pref, x_sorti2, x_sedge, x_redge, x_medge, x_gedge, x_etab, x_fan, cov_local;
    long long *h_cnt = nullptr;  // pinned, world*world + 4
};

namespace {

inline int grid_for(int64_t n, int threads) { return (int)std::max<int64_t>(1, (n + threads - 1) / threads); }

struct Phase {
    amira_gmg *h;
    int ph;
    Phase(amira_gmg *h_, int ph_) : h(h_), ph(ph_) {
        if (h->profiling) {
            cudaEventRecord(h->ev[ph][0], h->cur);
            h->ev_used[ph] = true;
        }
    }
    ~Phase() {
        if (h->profiling) cudaEventRecord(h->ev[ph][1], h->cur);
    }
};

#define LAUNCH(h, kern, grid, block, ...)                              \
    do {                                                               \
        kern<<<(grid), (block), 0, (h)->cur>>>(__VA_ARGS__);           \
        (h)->launches++;                                               \
        AMIRA_CUDA(cudaGetLastError());                                \
    } while (0)

// launches inside this scope go to the second stream
struct SideStream {
    amira_gmg *h;
    explicit SideStream(amira_gmg *h_) : h(h_) {
        static const bool one_stream = getenv("AMIRA_ONE_STREAM") != nullptr;  // developer experiments: clean per-phase times
        h->cur = one_stream ? h->stream : h->stream2;
    }
    ~SideStream() { h->cur = h->stream; }
};

inline long long *dsz(amira_gmg *h, int i) { return h->d_sizes.as<long long>() + i; }
inline Cnt dcnt(amira_gmg *h, int i) { return Cnt{dsz(h, i), 0}; }

inline int64_t scan_tiles(int64_t n_max) { return (n_max + 1 + SCAN_TILE - 1) / SCAN_TILE + 1; }

// exclusive scan over items 0..n (n on the device or immediate, at most n_max) on the current stream
template <typename L, typename S>
int run_scan(amira_gmg *h, L load, S store, const long long *n_ptr, long long n_mul, long long n_imm, int64_t n_max) {
    const int64_t tiles = scan_tiles(n_max);
    const size_t bytes = sizeof(unsigned long long) * (size_t)tiles;
    unsigned long long *state;
    if (h->scan_pool_used + bytes <= h->scan_pool_ready) {
        // inside a build: a piece of the pool the build cleared when it was enqueued
        state = reinterpret_cast<unsigned long long *>(static_cast<char *>(h->scan_pool.p) + h->scan_pool_used);
        h->scan_pool_used += bytes;
    } else {
        DevBuf &ws = h->scan_state[h->cur == h->stream2 ? 1 : 0];
        AMIRA_TRY(ws.reserve(bytes));  // reserved by reserve_graph; grows otherwise
        AMIRA_CUDA(cudaMemsetAsync(ws.p, 0, bytes, h->cur));
        h->lib_launches++;
        state = ws.as<unsigned long long>();
    }
    k_exscan<<<(unsigned int)(tiles - 1), SCAN_THREADS, 0, h->cur>>>(load, store, n_ptr, n_mul, n_imm, state);
    h->launches++;
    AMIRA_CUDA(cudaGetLastError());
    return AMIRA_OK;
}

// gene calls one GPU takes: positions inside the node -> reads transpose are 32-bit (shard the reads beyond that)
constexpr int64_t MAX_CALLS = 0xFFFF0000ll;

int bits_for64(int64_t n) {
    int b = 1;
    while (b < 62 && (1ll << b) < n) ++b;
    return b;
}

int bits_for_ids(unsigned int max_abs) {
    // |id| <= 2^(b-1) - 2: the all-ones and all-zero field values stay free
    int b = 2;
    while (b < 32 && ((1ull << (b - 1)) - 2) < (unsigned long long)max_abs) ++b;
    return b;
}

void reset_graph(amira_gmg *h) {
    h->n_nodes = h->n_edges = h->W = h->n_inc = h->n_short = h->n_fw = h->n_bw = h->n_comps = 0;
    h->pending = 0;
}

int sharded_merge_nodes(amira_gmg *h);
int sharded_merge_edges(amira_gmg *h);

// segmented sort on the current stream: segment s < *n_seg_ptr * mul has off[s+1] - off[s] keys below `max_value`;
// in place (a_start == nullptr, out_of_place == false: `a` sorted, `b` is scratch) or from a (segment starts
// a_start[s], or off[s]) into b
int run_segsort(amira_gmg *h, uint32_t *a, uint32_t *b, const int64_t *off, const uint32_t *a_start, bool out_of_place,
                const long long *n_seg_ptr, int mul, int64_t seg_max, int64_t elem_max, int64_t max_value, uint32_t *dups,
                unsigned long long *total_dups) {
    DevBuf &wb = h->seg_work[h->cur == h->stream2 ? 1 : 0];
    const int64_t cap = elem_max / SEG_BITONIC_MAX + 64;
    AMIRA_TRY(wb.reserve(sizeof(long long) * (size_t)(cap + 2)));  // reserved by reserve_graph; grows otherwise
    SegWork work{wb.as<unsigned int>(), wb.as<long long>() + 1, cap};
    AMIRA_CUDA(cudaMemsetAsync(wb.p, 0, sizeof(long long), h->cur));
    h->lib_launches++;
    const int bits = bits_for64(std::max<int64_t>(max_value, 2));
    SegJob J;
    J.a = a; J.b = b; J.off = off; J.a_start = a_start; J.n_seg_ptr = n_seg_ptr; J.seg_mul = mul;
    J.dups = dups; J.total_dups = total_dups;
    // the last pass must land in the destination: an even number of passes in place, an odd one out of place
    if (out_of_place) J.passes = bits <= 3 * 8 ? 3 : (bits <= 3 * SEG_MAX_DIGIT_BITS ? 3 : 5);
    else J.passes = bits <= 2 * SEG_MAX_DIGIT_BITS ? 2 : 4;
    J.digit_bits = std::max(5, (bits + J.passes - 1) / J.passes);
    const int grid_main = (int)std::min<int64_t>(grid_for(seg_max, 256), (int64_t)h->n_sm * 8);
    LAUNCH(h, k_segsort_main, grid_main, 256, J, work);
    LAUNCH(h, k_segsort_warp, (int)std::min<int64_t>((cap + 3) / 4, (int64_t)h->n_sm * 4), 128, J, work);
    // shared memory: the digit counters of 8 warps + two key buffers (8192 keys each when they fit ~72 KB)
    const size_t cnt_bytes = sizeof(unsigned int) * SEG_RADIX_WARPS * ((size_t)1 << J.digit_bits);
    const int kcap = 0;  // everything that fits shared memory is sorted by k_segsort_warp
    const size_t smem = cnt_bytes + 2 * sizeof(uint32_t) * (size_t)kcap;
    const int grid_rad = (int)std::min<int64_t>(cap, (int64_t)h->n_sm * 3);
    k_segsort_radix<<<grid_rad, SEG_RADIX_THREADS, smem, h->cur>>>(J, work, kcap);
    h->launches++;
    AMIRA_CUDA(cudaGetLastError());
    return AMIRA_OK;
}

// node -> forward/backward edge CSR from the current edge arrays (degrees already counted in adj_off
// when counted == true)
int build_adjacency(amira_gmg *h, bool counted) {
    Phase ph(h, AMIRA_PH_ADJACENCY);
    const Cnt N = dcnt(h, SZ_NODES), E = dcnt(h, SZ_EDGES);
    unsigned long long *deg = h->adj_off.as<unsigned long long>();
    if (!counted) {
        LAUNCH(h, k_fill_u64, h->n_sm * 4, 256, deg, N, 2, 2, 0ull);
        LAUNCH(h, k_adj_count, (int)std::min<int64_t>(grid_for(h->cap_edges, 256), (int64_t)h->n_sm * 32), 256, h->e_src.as<int32_t>(), h->e_sd.as<int8_t>(), E, N, deg);
    }
    // number of segments = 2N, on the device: the scan runs over 2N + 1 items
    AMIRA_TRY(run_scan(h, DegLoad{deg}, DegStore{h->adj_off.as<int64_t>(), h->adj_cursor.as<unsigned long long>(), N, dsz(h, 0)},
                       dsz(h, SZ_NODES), 2, 0, 2 * h->cap_nodes + 1));
    LAUNCH(h, k_adj_scatter, (int)std::min<int64_t>(grid_for(h->cap_edges, 256), (int64_t)h->n_sm * 32), 256, h->e_src.as<int32_t>(), h->e_sd.as<int8_t>(), E, N,
           h->adj_cursor.as<unsigned long long>(), h->adj_edges.as<uint32_t>());
    AMIRA_TRY(run_segsort(h, h->adj_edges.as<uint32_t>(), h->adj_tmp.as<uint32_t>(), h->adj_off.as<int64_t>(), nullptr, false,
                          dsz(h, SZ_NODES), 2, 2 * h->cap_nodes, h->cap_edges, h->cap_edges + 1, nullptr, nullptr));
    return AMIRA_OK;
}

// ---- build plan: table layout and every capacity, reserved before anything is enqueued (a buffer
// that grows synchronises the device; nothing below this point allocates) ------------------------------
int plan_build(amira_gmg *h) {
    const int64_t R = h->R, G = h->G;
    const int k = h->k;
    cudaStream_t st = h->stream;
    // Amira rebuilds the graph of (nearly) the same reads ~10-100x per sample: the previous build's
    // unique counts, scaled by the call-count ratio, size the tables; a cold build uses G/4 slots.
    // Either way an overflow is detected on the device and the build is redone larger.
    int64_t ncap = std::max<int64_t>(4096, G / 4), ecap = std::max<int64_t>(4096, G / 4);
    // Load factor: a warp waits for the longest probe sequence among its lanes, so the 16-byte node table runs
    // below 50 % load: 42 % (2.4 slots per expected node).  Measured on the C5 shard, whole build: 1.97 ms at 1.6
    // (62 %), 1.94 at 2.0, 1.92 at 2.4, 1.94 at 2.8, 1.98 at 3.2, 2.14 at 4.0 -- the insert kernel likes a sparse
    // table, every pass that scans the table and the L2 like a small one.  The edge table is insensitive and stays
    // at 50 %, as do the 32-byte layouts.
    if (h->id_bits == 0 && G > 0) {
        // first build on this handle: measure the largest |id| (later builds learn it from the insert kernel)
        if (h->n_pieces) AMIRA_CUDA(cudaStreamWaitEvent(st, h->ev_h2d[h->n_pieces - 1], 0));  // needs every id
        AMIRA_TRY(h->d_maxabs.reserve(2 * sizeof(unsigned int)));
        AMIRA_CUDA(cudaMemsetAsync(h->d_maxabs.p, 0, sizeof(unsigned int), st));
        LAUNCH(h, k_max_abs, std::min<int>(grid_for(G, 256), h->n_sm * 16), 256, h->ids, G, h->d_maxabs.as<unsigned int>());
        unsigned int max_abs = 0;
        AMIRA_CUDA(cudaMemcpyAsync(&max_abs, h->d_maxabs.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
        AMIRA_CUDA(cudaStreamSynchronize(st));
        h->id_bits = bits_for_ids(max_abs);
    }
    // Layout of the node table: a gene takes id_bits bits in a packed key.  k * id_bits <= 85: 16-byte slots
    // whose identity is the key itself; <= 124: 32-byte slots with the key published next to the claim
    // word; else gene-mers are compared through ids.
    const int T = k * (h->id_bits ? h->id_bits : 32);
    const bool n16 = T <= KEY16_BITS && h->id_bits > 0 && h->id_bits < 32 && !(h->force_layout & 1);
    h->key_bits = (T <= 124 && h->id_bits > 0 && h->id_bits < 32 && !(h->force_layout & 4)) ? h->id_bits : 0;
    const bool e16 = G < (1ll << ORD32_P_BITS) && !(h->force_layout & 2);
    double nslack = n16 ? 2.4 : 2.0, eslack = 2.0;
    if (const char *e = getenv("AMIRA_NODE_SLACK")) nslack = atof(e);  // developer experiments
    if (const char *e = getenv("AMIRA_EDGE_SLACK")) eslack = atof(e);
    if (h->hint_nodes > 0) ncap = h->hint_nodes * 2 + 1024;
    else if (h->prev_G > 0 && G <= 4 * h->prev_G)
        ncap = (int64_t)((double)h->prev_nodes * ((double)G / (double)h->prev_G) * nslack) + 4096;
    if (h->hint_edges > 0) ecap = h->hint_edges * 2 + 1024;
    else if (h->prev_G > 0 && G <= 4 * h->prev_G)
        ecap = (int64_t)((double)h->prev_und_edges * ((double)G / (double)h->prev_G) * eslack) + 4096;
    ncap = std::min<int64_t>(ncap * h->grow_n, 0x7FFFFFF0ll) & ~1ll;  // buckets of two slots
    ecap = std::min<int64_t>(ecap * h->grow_e, 0x3FFFFFF0ll) & ~1ll;
    h->n16 = n16;
    h->e16 = e16;
    h->ncap = (unsigned int)ncap;
    h->ecap = (unsigned int)ecap;
    const size_t nbytes = n16 ? (sizeof(NodeSlot16) + sizeof(unsigned int)) * (size_t)ncap : sizeof(NodeSlot) * (size_t)ncap;
    const size_t ebytes = (e16 ? sizeof(EdgeSlot16) : sizeof(EdgeSlot)) * (size_t)ecap;
    AMIRA_TRY(h->ntab.reserve(nbytes));
    AMIRA_TRY(h->etab.reserve(ebytes));
    AMIRA_TRY(h->slot_info.reserve(sizeof(uint2) * (size_t)(ncap + 1)));
    if (n16) {  // [slots][coverage]
        unsigned int *side = reinterpret_cast<unsigned int *>(h->ntab.as<NodeSlot16>() + ncap);
        h->nview = NodeView{h->ntab.as<unsigned long long>(), side, h->slot_info.as<uint2>(), 2, 1, h->ncap};
    } else {
        unsigned int *u = h->ntab.as<unsigned int>();
        h->nview = NodeView{h->ntab.as<unsigned long long>(), u + 2, h->slot_info.as<uint2>(), 4, 8, h->ncap};
    }
    h->eview = EdgeView{h->etab.p, h->ecap, e16 ? 1 : 0};

    const int64_t n_tiles = (G + INS_TILE - 1) / INS_TILE, n_words = (G + 31) / 32;
    const int64_t gcap = std::max<int64_t>(G, 1);
    AMIRA_TRY(h->win_off.reserve(sizeof(int64_t) * (R + 2)));
    AMIRA_TRY(h->is_short.reserve(R + 1));
    AMIRA_TRY(h->to_correct.reserve(R + 1));
    AMIRA_TRY(h->tile_r0.reserve(sizeof(int32_t) * (n_tiles + 1)));
    AMIRA_TRY(h->win_slot.reserve(sizeof(int32_t) * gcap + 32));
    AMIRA_TRY(h->win_node.reserve(sizeof(int32_t) * gcap + 32));
    AMIRA_TRY(h->win_dir.reserve(gcap));
    AMIRA_TRY(h->win_read.reserve(sizeof(int32_t) * gcap + 32));
    if (h->has_pos) {
        AMIRA_TRY(h->win_start.reserve(sizeof(int32_t) * gcap));
        AMIRA_TRY(h->win_end.reserve(sizeof(int32_t) * gcap));
    }
    AMIRA_TRY(h->bitmaps.reserve(sizeof(unsigned int) * 3 * (n_words + 1)));
    AMIRA_TRY(h->cnt_node.reserve(sizeof(int) * (n_words + 1)));
    AMIRA_TRY(h->cnt_edge.reserve(sizeof(int) * (n_words + 1)));
    return AMIRA_OK;
}

// node / edge arrays and the scratch of the passes after the insert, for at most capN nodes and capE
// directed edges (one GPU: the table capacities bound them; multi-GPU: the merged counts are known)
int reserve_graph(amira_gmg *h, int64_t capN, int64_t capE) {
    const int64_t G = std::max<int64_t>(h->G, 1), R = h->R, n_words = (h->G + 31) / 32;
    const int k = h->k;
    h->cap_nodes = capN;
    h->cap_edges = capE;
    AMIRA_TRY(h->node_key.reserve(sizeof(int32_t) * std::max<int64_t>(1, capN * k)));
    AMIRA_TRY(h->node_cov.reserve(sizeof(uint32_t) * (capN + 1)));
    AMIRA_TRY(h->node_dir.reserve(capN + 1));
    AMIRA_TRY(h->node_comp.reserve(sizeof(uint32_t) * (capN + 1)));
    AMIRA_TRY(h->parent.reserve(sizeof(int32_t) * (capN + 1)));
    AMIRA_TRY(h->link.reserve(capN + 2));
    if (h->prev_nodes > 0 && h->prev_nodes <= UF_SMALL_RUNS) AMIRA_TRY(h->run_pairs.reserve(sizeof(unsigned long long) * (size_t)(capE / 2 + 4)));
    AMIRA_TRY(h->run_id.reserve(sizeof(int32_t) * (capN + 2)));
    AMIRA_TRY(h->is_root.reserve(sizeof(int) * (capN + 2)));
    AMIRA_TRY(h->cc_min.reserve(sizeof(unsigned int) * (capN + 1)));
    AMIRA_TRY(h->reads_off.reserve(sizeof(int64_t) * (capN + 2)));
    AMIRA_TRY(h->dups.reserve(sizeof(uint32_t) * (capN + 1)));
    AMIRA_TRY(h->reads.reserve(sizeof(uint32_t) * G));
    AMIRA_TRY(h->e_src.reserve(sizeof(int32_t) * (capE + 2)));
    AMIRA_TRY(h->e_tgt.reserve(sizeof(int32_t) * (capE + 2)));
    AMIRA_TRY(h->e_sd.reserve(capE + 2));
    AMIRA_TRY(h->e_td.reserve(capE + 2));
    AMIRA_TRY(h->e_cov.reserve(sizeof(uint32_t) * (capE + 2)));
    AMIRA_TRY(h->adj_off.reserve(sizeof(int64_t) * (2 * capN + 3)));
    AMIRA_TRY(h->adj_cursor.reserve(sizeof(unsigned long long) * (2 * capN + 3)));
    AMIRA_TRY(h->adj_edges.reserve(sizeof(uint32_t) * (capE + 1)));
    AMIRA_TRY(h->adj_tmp.reserve(sizeof(uint32_t) * (capE + 1)));
    AMIRA_TRY(h->reads_tmp.reserve(sizeof(uint32_t) * G));
    AMIRA_TRY(h->inc_rec.reserve(sizeof(uint2) * (size_t)G));
    {
        // units of the node -> reads transpose: upper bound from the call count and the node capacity; more than
        // INC_NB_MAX of them share buckets (a unit then sweeps its whole bucket)
        UnitPlan &u = h->unit_plan;
        const int64_t n_max = h->G / INC_C + std::min<int64_t>(capN, h->world > 1 ? capN : std::max<int64_t>(h->G, 1)) / INC_S + 2;
        u.nb_max = (n_max <= INC_NB_MAX && !(h->force_layout & 8)) ? INC_NB_MAX : INC_NB_BIG;
        u.g = (h->force_layout & 16) ? 2 : 0;
        while (((n_max + (1ll << u.g) - 1) >> u.g) > u.nb_max) ++u.g;
        u.n_buckets = (int)((n_max + (1ll << u.g) - 1) >> u.g);
        u.n_units = u.n_buckets << u.g;
        u.read_lo = (uint32_t)h->first_read_global;
        u.rscale = (uint32_t)(0xFFFFFFFFull / (unsigned long long)std::max<int64_t>(R, 1));
        AMIRA_TRY(h->unit_lo.reserve(sizeof(int) * ((size_t)u.n_units + 2)));
        AMIRA_TRY(h->bucket_cursor.reserve(sizeof(unsigned int) * 2 * INC_NB_BIG));  // cursors, then region starts
    }
    for (int i = 0; i < 2; ++i)  // either stream may sort either array (the filter rebuilds the adjacency on the main one)
        AMIRA_TRY(h->seg_work[i].reserve(sizeof(long long) * (size_t)(std::max<int64_t>(G, capE) / SEG_BITONIC_MAX + 64 + 2)));
    const int64_t scan_max = std::max<int64_t>(std::max<int64_t>(R + 2, n_words + 2), std::max<int64_t>(2 * capN + 3, capE + 2));
    for (int i = 0; i < 2; ++i) AMIRA_TRY(h->scan_state[i].reserve(sizeof(unsigned long long) * (size_t)scan_tiles(scan_max)));
    return AMIRA_OK;
}

// status + sizes -> pinned host memory; which = 0: early copy (after the tables are final), 1: final copy
int enqueue_report(amira_gmg *h, int which) {
    AMIRA_CUDA(cudaMemcpyAsync(h->h_status + which * ST_COUNT, h->d_status.p, sizeof(int) * ST_COUNT, cudaMemcpyDeviceToHost,
                               h->stream));
    AMIRA_CUDA(cudaMemcpyAsync(h->h_sizes + which * SZ_COUNT, h->d_sizes.p, sizeof(long long) * SZ_COUNT,
                               cudaMemcpyDeviceToHost, h->stream));
    if (!h->capturing) AMIRA_CUDA(cudaEventRecord(which ? h->ev_done : h->ev_early, h->stream));  // (a replayed graph: recorded after the launch)
    h->lib_launches += 2;
    return AMIRA_OK;
}

// ---- windows + insert: per-read pass, window offsets, hash tables ----------------------------------
int enqueue_insert(amira_gmg *h) {
    const int64_t R = h->R, G = h->G;
    const int k = h->k;
    cudaStream_t st = h->stream;
    const int64_t n_tiles = (G + INS_TILE - 1) / INS_TILE;
    AMIRA_CUDA(cudaMemsetAsync(h->d_status.p, 0, sizeof(int) * ST_COUNT, st));
    AMIRA_CUDA(cudaMemsetAsync(h->d_sizes.p, 0, sizeof(long long) * SZ_COUNT, st));
    h->lib_launches += 2;
    h->scan_pool_used = h->scan_pool_ready = 0;
    if (h->world == 1) {
        // the seven scans of a one-GPU build (window offsets, first-seen ranks, runs, degrees, component firsts,
        // read offsets + slack) share one cleared pool
        const int64_t n_words = (G + 31) / 32;
        const size_t need = sizeof(unsigned long long) * (size_t)(scan_tiles(R) + scan_tiles(n_words) + 3 * scan_tiles(h->cap_nodes) +
                                                                  scan_tiles(2 * h->cap_nodes + 1) + 8);
        AMIRA_TRY(h->scan_pool.reserve(need));
        AMIRA_CUDA(cudaMemsetAsync(h->scan_pool.p, 0, need, st));
        h->lib_launches++;
        h->scan_pool_ready = need;
    }
    {
        Phase ph(h, AMIRA_PH_WINDOWS);
        LAUNCH(h, k_read_windows, grid_for(R + 1, 256), 256, h->off, R, k, G, h->win_off.as<int64_t>(),
               h->is_short.as<uint8_t>(), h->to_correct.as<uint8_t>(), h->tile_r0.as<int32_t>(),
               h->d_sizes.as<long long>(), h->d_status.as<int>());
        AMIRA_TRY(run_scan(h, WinOffLoad{h->win_off.as<int64_t>()},
                           WinOffStore{h->win_off.as<int64_t>(), R, dsz(h, 0)}, nullptr, 1, R, R));
    }
    Phase ph(h, AMIRA_PH_INSERT);
    const size_t nbytes = h->n16 ? (sizeof(NodeSlot16) + sizeof(unsigned int)) * (size_t)h->ncap : sizeof(NodeSlot) * (size_t)h->ncap;
    const size_t ebytes = (h->e16 ? sizeof(EdgeSlot16) : sizeof(EdgeSlot)) * (size_t)h->ecap;
    AMIRA_CUDA(cudaMemsetAsync(h->ntab.p, 0xFF, nbytes, st));
    AMIRA_CUDA(cudaMemsetAsync(h->etab.p, 0xFF, ebytes, st));
    h->lib_launches += 2;
    if (n_tiles == 0) return AMIRA_OK;
    BuildParams P;
    P.ids = h->ids; P.off = h->off; P.win_off = h->win_off.as<int64_t>();
    P.tile_r0 = h->tile_r0.as<int32_t>(); P.ps = h->ps; P.pe = h->pe;
    P.G = G; P.R = R; P.n_tiles = n_tiles; P.k = k;
    P.tile_lo = 0; P.tile_hi = n_tiles;
    P.ntab = h->ntab.as<NodeSlot>(); P.ntab16 = h->ntab.as<NodeSlot16>(); P.ncov = h->nview.cov;
    P.ncap = h->ncap; P.etab = h->etab.as<EdgeSlot>(); P.etab16 = h->etab.as<EdgeSlot16>(); P.ecap = h->ecap;
    P.win_node = h->win_slot.as<int32_t>(); P.win_dir = h->win_dir.as<int8_t>();
    P.win_read = h->win_read.as<int32_t>();
    P.win_start = h->has_pos ? h->win_start.as<int32_t>() : nullptr;
    P.win_end = h->has_pos ? h->win_end.as<int32_t>() : nullptr;
    P.status = h->d_status.as<int>();
    P.read_base = h->first_read_global;
    P.key_bits = h->key_bits;
    P.ids_aligned = (reinterpret_cast<uintptr_t>(h->ids) & 15) == 0;
    h->local_P = P;
    const bool n16 = h->n16, e16 = h->e16;
    {
        Phase phk(h, AMIRA_PH_INSERT_KERNEL);
#define INSERT_KE(KK, NN, EE) LAUNCH(h, (k_insert_windows<KK, NN, EE>), grid, INS_THREADS, P)
#define INSERT_K(KK)                                  \
    do {                                              \
        if (n16 && e16) INSERT_KE(KK, true, true);    \
        else if (n16) INSERT_KE(KK, true, false);     \
        else if (e16) INSERT_KE(KK, false, true);     \
        else INSERT_KE(KK, false, false);             \
    } while (0)
        // one launch over everything, or (host input still streaming in) one launch per piece:
        // piece i's chunks minus its last one, which needs the first ids of piece i+1
        const int n_launch = std::max(1, h->n_pieces);
        int64_t lo = 0;
        for (int piece = 0; piece < n_launch; ++piece) {
            int64_t hi = n_tiles;
            if (h->n_pieces) {
                AMIRA_CUDA(cudaStreamWaitEvent(st, h->ev_h2d[piece], 0));
                if (piece + 1 < n_launch) hi = std::max<int64_t>(lo, h->piece_end[piece] / INS_TILE - 1);
            }
            P.tile_lo = lo;
            P.tile_hi = hi;
            lo = hi;
            if (P.tile_hi <= P.tile_lo) continue;
            const int grid = (int)std::min<int64_t>((P.tile_hi - P.tile_lo + INS_WARPS - 1) / INS_WARPS,
                                                    (int64_t)h->n_sm * h->insert_ctas_per_sm);
            if (k == 3) INSERT_K(3);
            else if (k == 5) INSERT_K(5);
            else if (k == 7) INSERT_K(7);
            else INSERT_K(0);
        }
#undef INSERT_K
#undef INSERT_KE
    }
    if (n_tiles > 1) {
        if (e16) LAUNCH(h, k_boundary_edges<true>, grid_for(n_tiles - 1, 256), 256, P);
        else LAUNCH(h, k_boundary_edges<false>, grid_for(n_tiles - 1, 256), 256, P);
    }
    return AMIRA_OK;
}

// ---- one GPU: first-seen ranks of nodes and edges, node arrays ------------------------------------
int enqueue_order(amira_gmg *h) {
    const int64_t G = h->G, n_words = (G + 31) / 32;
    cudaStream_t st = h->stream;
    unsigned int *bm_node = h->bitmaps.as<unsigned int>();
    unsigned int *bm_ea = bm_node + (n_words + 1), *bm_eb = bm_ea + (n_words + 1);
    {
        Phase ph(h, AMIRA_PH_ORDER);
        AMIRA_CUDA(cudaMemsetAsync(h->bitmaps.p, 0, sizeof(unsigned int) * 3 * (n_words + 1), st));
        h->lib_launches++;
        const unsigned int tmax = std::max(h->ncap, h->ecap);
        LAUNCH(h, k_mark_first, std::min<int>(grid_for(tmax, 256), h->n_sm * 16), 256, h->nview, h->eview, bm_node, bm_ea, bm_eb);
        AMIRA_TRY(run_scan(h, RankLoad{bm_node, bm_ea, bm_eb},
                           RankStore{h->cnt_node.as<int>(), h->cnt_edge.as<int>(), n_words, dsz(h, 0), h->d_status.as<int>()}, nullptr, 1, n_words,
                           n_words));
    }
    AMIRA_TRY(enqueue_report(h, 0));
    {
        Phase ph(h, AMIRA_PH_EMIT_NODES);
        // (node -> slot lives in is_root, which the components pass only needs later)
        LAUNCH(h, k_rank_nodes, std::min<int>(grid_for(h->ncap, 256), h->n_sm * 16), 256, h->nview, bm_node, h->cnt_node.as<int>(),
               h->is_root.as<uint32_t>());
        LAUNCH(h, k_emit_nodes, (int)std::min<int64_t>(grid_for(h->cap_nodes, 256), (int64_t)h->n_sm * 16), 256, h->nview, h->ids, h->k,
               dcnt(h, SZ_NODES), h->is_root.as<uint32_t>(), h->node_key.as<int32_t>(), h->node_cov.as<uint32_t>(),
               h->node_dir.as<int8_t>(), h->link.as<uint8_t>(),
               (h->n16 && h->key_bits > 0) ? h->ntab.as<NodeSlot16>() : (const NodeSlot16 *)nullptr, h->key_bits);
    }
    return AMIRA_OK;
}

// ---- the passes after the node order is known -------------------------------------------------------
// branch B (second stream): edges in first-seen order, union-find, adjacency, components
// branch A (main stream):   per-read node lists + node -> reads scatter, segment sort
// branch B, on the current stream (the caller has switched to the second one)
int enqueue_tail_side(amira_gmg *h) {
    const int64_t G = h->G, n_words = (G + 31) / 32;
    const Cnt N = dcnt(h, SZ_NODES), E = dcnt(h, SZ_EDGES);
    unsigned int *bm_node = h->bitmaps.as<unsigned int>();
    unsigned int *bm_ea = bm_node + (n_words + 1), *bm_eb = bm_ea + (n_words + 1);
    {
        unsigned long long *deg = h->adj_off.as<unsigned long long>();
        bool counted = false;
        const int32_t *run_ids = nullptr;
        if (h->world == 1) {
            Phase ph(h, AMIRA_PH_EMIT);
            LAUNCH(h, k_fill_u64, h->n_sm * 4, 256, deg, N, 2, 2, 0ull);
            // (directed edge -> table entry lives in adj_tmp, which the adjacency pass only needs later)
            LAUNCH(h, k_rank_edges, std::min<int>(grid_for(h->ecap, 256), h->n_sm * 16), 256, h->eview, bm_ea, bm_eb,
                   h->cnt_edge.as<int>(), h->adj_tmp.as<uint32_t>(), h->d_status.as<int>());
            LAUNCH(h, k_emit_edges, (int)std::min<int64_t>(grid_for(h->cap_edges, 256), (int64_t)h->n_sm * 16), 256, h->eview, h->nview,
                   h->adj_tmp.as<uint32_t>(), E, N, h->e_src.as<int32_t>(), h->e_tgt.as<int32_t>(), h->e_sd.as<int8_t>(),
                   h->e_td.as<int8_t>(), h->e_cov.as<uint32_t>(), deg, h->link.as<uint8_t>());
            counted = true;
            // runs of consecutive first-seen nodes joined by an edge (a prefix count, no pointer chasing), then
            // union-find over the runs with the edges that leave a run, in first-seen edge order
            run_ids = h->run_id.as<int32_t>();
            AMIRA_TRY(run_scan(h, RunLoad{h->link.as<uint8_t>()}, RunStore{h->run_id.as<int32_t>(), h->parent.as<int32_t>(), N},
                               dsz(h, SZ_NODES), 1, 0, h->cap_nodes));
            // (measured SLOWER than this in-order scan of the edge arrays with ~4 of 32 lanes in a find, 0.19 ms: a compacted
            // list of the run-leaving edges with every lane busy, 0.38 ms; hanging every run under its smallest
            // neighbour run + pointer jumping first, 0.27 ms with hashed linking and 0.51 ms with linking by index)
            const unsigned long long *done = nullptr;
            if (h->prev_nodes > 0 && h->prev_nodes <= UF_SMALL_RUNS) {
                // small graph (by the previous build on this handle; the kernels check the real run count): unions at
                // shared-memory latency.  pairs[0] = list length, pairs[1] = done flag, then the list.
                unsigned long long *pairs = h->run_pairs.as<unsigned long long>();
                AMIRA_CUDA(cudaMemsetAsync(pairs, 0, 2 * sizeof(unsigned long long), h->cur));
                h->lib_launches++;
                LAUNCH(h, k_collect_run_edges, (int)std::min<int64_t>(grid_for(h->cap_edges, 256), (int64_t)h->n_sm * 16), 256, h->e_src.as<int32_t>(),
                       h->e_tgt.as<int32_t>(), E, N, run_ids, pairs + 2, pairs);
                k_union_small<<<1, UF_SMALL_THREADS, sizeof(int32_t) * UF_SMALL_RUNS, h->cur>>>(pairs + 2, pairs, N, run_ids, h->parent.as<int32_t>(), pairs + 1);
                h->launches++;
                AMIRA_CUDA(cudaGetLastError());
                done = pairs + 1;
            }
            LAUNCH(h, k_union_edges, (int)std::min<int64_t>(grid_for(h->cap_edges, 256), (int64_t)h->n_sm * 64), 256, h->e_src.as<int32_t>(), h->e_tgt.as<int32_t>(), E, h->parent.as<int32_t>(), run_ids, done);
        } else if (h->sh_Eg > 0) {
            Phase ph(h, AMIRA_PH_EMIT);
            LAUNCH(h, k_emit_edges_sorted, grid_for(h->sh_Eg, 256), 256, h->x_sorti2.as<unsigned int>(), h->sh_gedge,
                   h->x_fan.as<int>(), (long long)h->sh_Eg, h->e_src.as<int32_t>(), h->e_tgt.as<int32_t>(),
                   h->e_sd.as<int8_t>(), h->e_td.as<int8_t>(), h->e_cov.as<uint32_t>(), h->link.as<uint8_t>());
        }
        if (h->world > 1) {
            run_ids = h->run_id.as<int32_t>();
            AMIRA_TRY(run_scan(h, RunLoad{h->link.as<uint8_t>()}, RunStore{h->run_id.as<int32_t>(), h->parent.as<int32_t>(), N},
                               dsz(h, SZ_NODES), 1, 0, h->cap_nodes));
            LAUNCH(h, k_union_edges, (int)std::min<int64_t>(grid_for(std::max<int64_t>(h->cap_edges, 1), 256), (int64_t)h->n_sm * 64), 256, h->e_src.as<int32_t>(), h->e_tgt.as<int32_t>(), E, h->parent.as<int32_t>(), run_ids, nullptr);
        }
        AMIRA_TRY(build_adjacency(h, counted));
        {
            Phase ph(h, AMIRA_PH_COMPONENTS);
            LAUNCH(h, k_fill_u32, h->n_sm * 4, 256, h->cc_min.as<uint32_t>(), N, 1, 1, 0xFFFFFFFFu);
            LAUNCH(h, k_cc_flatten, (int)std::min<int64_t>(grid_for(h->cap_nodes, 256), (int64_t)h->n_sm * 64), 256, h->parent.as<int32_t>(), N, h->cc_min.as<unsigned int>(),
                   h->node_comp.as<uint32_t>(), run_ids);
            AMIRA_TRY(run_scan(h, FirstLoad{h->node_comp.as<uint32_t>(), h->cc_min.as<unsigned int>()},
                               FirstStore{h->is_root.as<int>(), N, dsz(h, 0)}, dsz(h, SZ_NODES), 1, 0, h->cap_nodes));
            LAUNCH(h, k_cc_number, (int)std::min<int64_t>(grid_for(h->cap_nodes, 256), (int64_t)h->n_sm * 64), 256, h->cc_min.as<unsigned int>(), h->is_root.as<int>(), N,
                   h->node_comp.as<uint32_t>());
        }
        AMIRA_CUDA(cudaEventRecord(h->ev_join, h->cur));
    }
    return AMIRA_OK;
}

// branch A, on the main stream
int enqueue_tail_main(amira_gmg *h) {
    const int64_t G = h->G;
    cudaStream_t st = h->stream;
    const Cnt N = dcnt(h, SZ_NODES);
    {
        // node -> reads (incidence.cuh): coverage per node (counted by the insert kernel) -> offsets, units,
        // records dealt into buckets (the same pass writes the per-read node lists), one CTA per unit
        const uint32_t *cov = h->world > 1 ? h->cov_local.as<uint32_t>() : h->node_cov.as<uint32_t>();
        const UnitPlan &u = h->unit_plan;
        {
            Phase ph(h, AMIRA_PH_REMAP);
            AMIRA_TRY(run_scan(h, CovLoad{cov}, CovStore{h->reads_off.as<int64_t>(), N, dsz(h, 0)}, dsz(h, SZ_NODES), 1, 0,
                               h->cap_nodes));
            LAUNCH(h, k_unit_table, (int)std::min<int64_t>(grid_for(std::max<int64_t>(h->ncap, h->cap_nodes + 1), 256), (int64_t)h->n_sm * 16), 256,
                   h->nview, h->reads_off.as<int64_t>(), dsz(h, SZ_NODES), u, h->unit_lo.as<int>(), h->d_status.as<int>());
            unsigned int *bcur = h->bucket_cursor.as<unsigned int>();
            LAUNCH(h, k_bucket_base, u.nb_max / 256, 256, h->unit_lo.as<int>(), h->reads_off.as<int64_t>(), u, bcur + INC_NB_BIG, bcur);
            // low coverage (by the previous build on this handle): large tiles, see incidence.cuh
            const bool wide = h->prev_nodes > 0 && h->prev_G < (int64_t)PART_WIDE_BELOW * h->prev_nodes;
            if (u.nb_max == INC_NB_MAX && !wide) {
                const int pgrid = (int)std::min<int64_t>(std::max<int64_t>(1, (G + PartSmall::TILE - 1) / PartSmall::TILE), (int64_t)h->n_sm * PartSmall::CTAS);
                k_partition<PartSmall><<<pgrid, PartSmall::THREADS, PartSmall::SMEM, st>>>(
                    h->slot_info.as<uint2>(), h->win_slot.as<int32_t>(), h->win_read.as<int32_t>(), h->win_node.as<int32_t>(),
                    (const long long *)h->d_sizes.p, bcur + INC_NB_BIG, u, bcur, h->inc_rec.as<uint2>());
            } else if (u.nb_max == INC_NB_MAX) {
                const int pgrid = (int)std::min<int64_t>(std::max<int64_t>(1, (G + PartWide::TILE - 1) / PartWide::TILE), (int64_t)h->n_sm * PartWide::CTAS);
                k_partition<PartWide><<<pgrid, PartWide::THREADS, PartWide::SMEM, st>>>(
                    h->slot_info.as<uint2>(), h->win_slot.as<int32_t>(), h->win_read.as<int32_t>(), h->win_node.as<int32_t>(),
                    (const long long *)h->d_sizes.p, bcur + INC_NB_BIG, u, bcur, h->inc_rec.as<uint2>());
            } else {
                const int pgrid = (int)std::min<int64_t>(std::max<int64_t>(1, (G + PartBig::TILE - 1) / PartBig::TILE), (int64_t)h->n_sm * PartBig::CTAS);
                k_partition<PartBig><<<pgrid, PartBig::THREADS, PartBig::SMEM, st>>>(
                    h->slot_info.as<uint2>(), h->win_slot.as<int32_t>(), h->win_read.as<int32_t>(), h->win_node.as<int32_t>(),
                    (const long long *)h->d_sizes.p, bcur + INC_NB_BIG, u, bcur, h->inc_rec.as<uint2>());
            }
            h->launches++;
            AMIRA_CUDA(cudaGetLastError());
        }
        if (!h->capturing) AMIRA_CUDA(cudaEventRecord(h->ev_reads_ready, st));
        Phase ph(h, AMIRA_PH_INCIDENCE);
        // in-place job over `reads` for the units that outgrow shared memory (and the lists they leave to the
        // work-list kernels of segsort.cuh)
        DevBuf &wb = h->seg_work[0];
        const int64_t wcap = std::max<int64_t>(G, 1) / SEG_BITONIC_MAX + 64;
        SegWork work{wb.as<unsigned int>(), wb.as<long long>() + 1, wcap};
        AMIRA_CUDA(cudaMemsetAsync(wb.p, 0, sizeof(long long), st));
        h->lib_launches++;
        const int64_t reads_global = h->world > 1 ? 0x7FFFFFF0ll : h->R;
        const int bits = bits_for64(std::max<int64_t>(reads_global + 1, 2));
        SegJob J;
        J.a = h->reads.as<uint32_t>(); J.b = h->reads_tmp.as<uint32_t>(); J.off = h->reads_off.as<int64_t>(); J.a_start = nullptr;
        J.n_seg_ptr = dsz(h, SZ_NODES); J.seg_mul = 1;
        J.dups = h->dups.as<uint32_t>(); J.total_dups = (unsigned long long *)dsz(h, SZ_DUPS);
        J.passes = bits <= 2 * SEG_MAX_DIGIT_BITS ? 2 : 4;
        J.digit_bits = std::max(5, (bits + J.passes - 1) / J.passes);
        k_unit_lists<<<u.n_units, INC_THREADS, INC_SMEM, st>>>(h->inc_rec.as<uint2>(), h->unit_lo.as<int>(), u, J, work);
        h->launches++;
        AMIRA_CUDA(cudaGetLastError());
        LAUNCH(h, k_segsort_warp, (int)std::min<int64_t>((wcap + 3) / 4, (int64_t)h->n_sm * 4), 128, J, work);
        const size_t cnt_bytes = sizeof(unsigned int) * SEG_RADIX_WARPS * ((size_t)1 << J.digit_bits);
        k_segsort_radix<<<(int)std::min<int64_t>(wcap, (int64_t)h->n_sm * 3), SEG_RADIX_THREADS, cnt_bytes, st>>>(J, work, 0);
        h->launches++;
        AMIRA_CUDA(cudaGetLastError());
    }
    return AMIRA_OK;
}

int enqueue_join(amira_gmg *h) {
    AMIRA_CUDA(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
    AMIRA_TRY(enqueue_report(h, 1));
    h->pending = 2;
    h->pending_is_build = true;
    return AMIRA_OK;
}

int enqueue_tail(amira_gmg *h) {
    AMIRA_CUDA(cudaEventRecord(h->ev_fork, h->stream));
    AMIRA_CUDA(cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
    {
        SideStream side(h);
        AMIRA_TRY(enqueue_tail_side(h));
    }
    AMIRA_TRY(enqueue_tail_main(h));
    return enqueue_join(h);
}

// (a negative count leaves the size alone)
__global__ void k_set_sizes(long long *sizes, long long n_nodes, long long n_edges) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        if (n_nodes >= 0) sizes[SZ_NODES] = n_nodes;
        if (n_edges >= 0) sizes[SZ_EDGES] = n_edges;
    }
}

int do_build(amira_gmg *h) {
    cudaStream_t st = h->stream;
    if (h->world == 1) {
        AMIRA_TRY(plan_build(h));
        AMIRA_TRY(reserve_graph(h, h->ncap, 2 * (int64_t)h->ecap));
        const amira_gmg::GraphKey key{h->ids, h->off, h->ps, h->pe, h->R, h->G, h->cap_nodes, h->cap_edges, h->ncap, h->ecap,
                                      h->k, h->key_bits, (h->n16 ? 1 : 0) | (h->e16 ? 2 : 0), buffer_generation().load()};
        static const bool no_graph = getenv("AMIRA_NO_GRAPH") != nullptr;
        const bool can_graph = h->input_on_device && !h->profiling && h->n_pieces == 0 && h->G <= (64ll << 20) && !no_graph;
        auto after_launch = [&]() -> int {
            AMIRA_CUDA(cudaEventRecord(h->ev_reads_ready, st));
            AMIRA_CUDA(cudaEventRecord(h->ev_early, st));
            AMIRA_CUDA(cudaEventRecord(h->ev_done, st));
            h->pending = 2;
            h->pending_is_build = true;
            h->graph_launches++;
            return AMIRA_OK;
        };
        if (can_graph && h->graph_exec && key == h->graph_key) {
            AMIRA_CUDA(cudaGraphLaunch(h->graph_exec, st));
            h->launches += h->graph_kernels;
            return after_launch();
        }
        if (can_graph && key == h->last_key) {
            if (h->graph_exec) {
                cudaGraphExecDestroy(h->graph_exec);
                h->graph_exec = nullptr;
            }
            AMIRA_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            h->capturing = true;
            const int64_t launches0 = h->launches;
            int rc = enqueue_insert(h);
            if (rc == AMIRA_OK) rc = enqueue_order(h);
            if (rc == AMIRA_OK) rc = enqueue_tail(h);
            h->capturing = false;
            cudaGraph_t graph = nullptr;
            const cudaError_t ce = cudaStreamEndCapture(st, &graph);
            if (rc == AMIRA_OK && ce == cudaSuccess && graph) {
                if (cudaGraphInstantiate(&h->graph_exec, graph, 0) != cudaSuccess) h->graph_exec = nullptr;
            }
            if (graph) cudaGraphDestroy(graph);
            if (h->graph_exec) {
                h->graph_key = key;
                h->graph_kernels = h->launches - launches0;
                AMIRA_CUDA(cudaGraphLaunch(h->graph_exec, st));
                return after_launch();
            }
            cudaGetLastError();  // capture failed: fall through to the plain launches
            h->pending = 0;
        }
        h->last_key = key;
        AMIRA_TRY(enqueue_insert(h));
        AMIRA_TRY(enqueue_order(h));
        return enqueue_tail(h);
    }
    // multi-GPU: the exchange needs host-side counts, so the local tables are finished synchronously
    for (int attempt = 0;; ++attempt) {
        AMIRA_TRY(plan_build(h));
        AMIRA_TRY(enqueue_insert(h));
        AMIRA_TRY(enqueue_report(h, 0));
        AMIRA_CUDA(cudaStreamSynchronize(st));
        const int *s = h->h_status;
        if (s[ST_ERR]) break;
        const bool unpack = s[ST_UNPACK] && h->key_bits > 0;
        if (unpack) h->id_bits = 0;
        if (!s[ST_OVERFLOW_N] && !s[ST_OVERFLOW_E] && !unpack) break;
        if (attempt >= 6) {
            set_error("hash tables overflowed after %d attempts (ncap=%u ecap=%u)", attempt + 1, h->ncap, h->ecap);
            return AMIRA_E_NOMEM;
        }
        if (s[ST_OVERFLOW_N]) h->grow_n *= 4;
        if (s[ST_OVERFLOW_E]) h->grow_e *= 4;
    }
    h->grow_n = h->grow_e = 1;
    if ((unsigned int)h->h_status[ST_MAXABS] > 0 && h->id_bits != 0) h->id_bits = bits_for_ids((unsigned int)h->h_status[ST_MAXABS]);
    // every rank must leave the build together: agree on the error status before any exchange
    AMIRA_TRY(comm_allreduce_max_i32(h->comm, h->d_status.as<int>(), 4, st));
    AMIRA_CUDA(cudaMemcpyAsync(h->h_status, h->d_status.p, sizeof(int) * ST_COUNT, cudaMemcpyDeviceToHost, st));
    AMIRA_CUDA(cudaStreamSynchronize(st));
    if (h->h_status[ST_ERR]) {
        const int e = h->h_status[ST_ERR];
        if (e == AMIRA_E_PALINDROME) set_error("Gene-mer and reverse complement gene-mer are identical");
        else set_error("invalid read offsets");
        return e;
    }
    h->W = h->h_sizes[SZ_W];
    h->n_short = h->h_sizes[SZ_SHORT];
    h->prev_G = h->G;
    // nodes first (main stream); then the per-read passes start on the main stream while the edges are exchanged,
    // merged and emitted on the second one
    AMIRA_TRY(sharded_merge_nodes(h));
    LAUNCH(h, k_set_sizes, 1, 32, h->d_sizes.as<long long>(), (long long)h->n_nodes, -1ll);
    AMIRA_CUDA(cudaEventRecord(h->ev_fork, st));
    AMIRA_CUDA(cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
    AMIRA_TRY(enqueue_tail_main(h));
    {
        SideStream side(h);
        AMIRA_TRY(sharded_merge_edges(h));
        LAUNCH(h, k_set_sizes, 1, 32, h->d_sizes.as<long long>(), -1ll, (long long)h->n_edges);
        AMIRA_TRY(enqueue_tail_side(h));
    }
    return enqueue_join(h);
}

// lazy removal of duplicate incidences (a gene-mer twice on one read), when the build counted any
int finalize_incidence(amira_gmg *h) {
    const int64_t N = h->n_nodes;
    const Cnt cn{nullptr, N};
    AMIRA_TRY(h->reads_off2.reserve(sizeof(int64_t) * (N + 2)));
    AMIRA_TRY(h->reads2.reserve(sizeof(uint32_t) * std::max<int64_t>(1, h->n_inc)));
    AMIRA_TRY(run_scan(h, UniqLoad{h->reads_off.as<int64_t>(), h->dups.as<uint32_t>()},
                       OffStore{h->reads_off2.as<int64_t>(), cn, dsz(h, SZ_INC)}, nullptr, 1, N, N));
    LAUNCH(h, k_compact_unique, (int)std::min<int64_t>(grid_for(N * 32, 256), (int64_t)h->n_sm * 8), 256,
           h->reads_off.as<int64_t>(), h->reads.as<uint32_t>(), h->reads_off2.as<int64_t>(), h->reads2.as<uint32_t>(), cn);
    long long n_inc = 0;
    AMIRA_CUDA(cudaMemcpyAsync(&n_inc, dsz(h, SZ_INC), sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    std::swap(h->reads_off, h->reads_off2);
    std::swap(h->reads, h->reads2);
    h->n_inc = n_inc;
    return AMIRA_OK;
}

// Wait for what the last build / filter reported and act on it.  early: only the counts that are known
// once the tables are final (nodes, edges, windows, short reads) are needed.
int finish(amira_gmg *h, bool early) {
    while (h->pending) {
        if (early && h->pending == 1) return h->last_status;
        const int which = (early && h->pending_is_build && h->world == 1) ? 0 : 1;
        AMIRA_CUDA(cudaEventSynchronize(which ? h->ev_done : h->ev_early));
        const int *s = h->h_status + which * ST_COUNT;
        const long long *z = h->h_sizes + which * SZ_COUNT;
        if (h->pending_is_build && h->world == 1) {
            // problems the device found: redo the build (synchronously from here on)
            const bool unpack = s[ST_UNPACK] && h->key_bits > 0;
            if (s[ST_ERR] || s[ST_STALE] || s[ST_OVERFLOW_N] || s[ST_OVERFLOW_E] || unpack) {
                AMIRA_CUDA(cudaEventSynchronize(h->ev_done));
                h->pending = 0;
                if (s[ST_STALE]) {
                    int64_t G = 0;
                    AMIRA_CUDA(cudaMemcpyAsync(&G, h->off + h->R, sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
                    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
                    if (G < 0 || G >= MAX_CALLS) {
                        set_error("bad call count %lld", (long long)G);
                        h->built = false;
                        return h->last_status = AMIRA_E_ARG;
                    }
                    h->G = h->cache_G = G;
                } else if (s[ST_ERR]) {
                    const int e = s[ST_ERR];
                    if (e == AMIRA_E_PALINDROME) set_error("Gene-mer and reverse complement gene-mer are identical");
                    else set_error("invalid read offsets");
                    h->built = false;
                    h->grow_n = h->grow_e = 1;
                    return h->last_status = e;
                } else {
                    if (++h->attempts > 6) {
                        set_error("hash tables overflowed after %d attempts (ncap=%u ecap=%u)", h->attempts, h->ncap, h->ecap);
                        h->built = false;
                        return h->last_status = AMIRA_E_NOMEM;
                    }
                    if (unpack) h->id_bits = 0;  // an id outgrew the remembered width: measure again
                    if (s[ST_OVERFLOW_N]) h->grow_n *= 4;
                    if (s[ST_OVERFLOW_E]) h->grow_e *= 4;
                }
                const int rc = do_build(h);
                if (rc != AMIRA_OK) {
                    h->built = false;
                    return h->last_status = rc;
                }
                continue;
            }
        }
        h->n_nodes = z[SZ_NODES];
        h->n_edges = z[SZ_EDGES];
        h->W = z[SZ_W];
        if (h->pending_is_build) h->n_short = z[SZ_SHORT];
        if (which == 0) {
            h->pending = 1;
            return h->last_status;
        }
        h->n_inc = z[SZ_INC];
        h->n_fw = z[SZ_FW];
        h->n_bw = h->n_edges - h->n_fw;
        // upper bound on component ids: ids are <= the number of nodes of the BUILD, and filters keep the ids
        if (h->pending_is_build) h->n_comps = h->n_nodes;
        h->pending = 0;
        if (h->pending_is_build) {
            if (h->world == 1) {
                h->prev_G = h->G;
                h->prev_nodes = h->n_nodes;
                h->prev_und_edges = (h->n_edges + 1) / 2 + 1;  // directed edges come in pairs, self-edges alone
                h->grow_n = h->grow_e = 1;
                h->attempts = 0;
                // the key width follows the data in both directions
                if (h->id_bits != 0 && (unsigned int)s[ST_MAXABS] > 0) h->id_bits = bits_for_ids((unsigned int)s[ST_MAXABS]);
            }
            if (z[SZ_DUPS] > 0) AMIRA_TRY(finalize_incidence(h));
        }
    }
    return h->last_status;
}

// everything a filter / node removal touches, reserved before its kernels are enqueued
int filter_reserve(amira_gmg *h) {
    if (!h->built) {
        set_error("filter before build");
        return AMIRA_E_STATE;
    }
    AMIRA_TRY(finish(h, false));
    if (!h->built) return h->last_status;
    const int64_t N = h->n_nodes, E = h->n_edges;
    const int k = h->k;
    AMIRA_TRY(h->keep_n.reserve(sizeof(int) * 2 * (N + 2)));
    AMIRA_TRY(h->keep_e.reserve(sizeof(int) * 2 * (E + 2)));
    AMIRA_TRY(h->node_key2.reserve(sizeof(int32_t) * std::max<int64_t>(1, N * k)));
    AMIRA_TRY(h->node_cov2.reserve(sizeof(uint32_t) * (N + 1)));
    AMIRA_TRY(h->node_dir2.reserve(N + 1));
    AMIRA_TRY(h->node_comp2.reserve(sizeof(uint32_t) * (N + 1)));
    AMIRA_TRY(h->reads_off2.reserve(sizeof(int64_t) * (N + 2)));
    AMIRA_TRY(h->reads2.reserve(sizeof(uint32_t) * std::max<int64_t>(1, h->n_inc)));
    AMIRA_TRY(h->e_src2.reserve(sizeof(int32_t) * (E + 2)));
    AMIRA_TRY(h->e_tgt2.reserve(sizeof(int32_t) * (E + 2)));
    AMIRA_TRY(h->e_sd2.reserve(E + 2));
    AMIRA_TRY(h->e_td2.reserve(E + 2));
    AMIRA_TRY(h->e_cov2.reserve(sizeof(uint32_t) * (E + 2)));
    AMIRA_TRY(h->comp_max.reserve(sizeof(uint32_t) * (h->n_comps + 2)));
    // the graph only shrinks: the capacities of the build (or of the previous filter) still hold
    h->cap_nodes = std::max<int64_t>(h->cap_nodes, N);
    h->cap_edges = std::max<int64_t>(h->cap_edges, E);
    return AMIRA_OK;
}

// mode 0: filter_graph thresholds; mode 1: remove_low_coverage_components; mode 2: the keep flags of the nodes are
// already in keep_n (remove_node for every node whose flag is 0)
int do_filter(amira_gmg *h, int mode, uint32_t thr_node, uint32_t thr_edge) {
    AMIRA_TRY(filter_reserve(h));
    const int64_t N = h->n_nodes, E = h->n_edges, W = h->W;
    const int k = h->k;
    cudaStream_t st = h->stream;
    h->filt_N = N;
    h->filt_E = E;
    if (N == 0) return AMIRA_OK;
    Phase ph(h, AMIRA_PH_FILTER);
    int *keep_n = h->keep_n.as<int>(), *new_n = keep_n + (N + 2);
    int *keep_e = h->keep_e.as<int>(), *new_e = keep_e + (E + 2);
    if (mode == 1) {
        AMIRA_CUDA(cudaMemsetAsync(h->comp_max.p, 0, sizeof(uint32_t) * (h->n_comps + 2), st));
        LAUNCH(h, k_component_max, grid_for(N, 256), 256, h->node_cov.as<uint32_t>(), h->node_comp.as<uint32_t>(), N,
               h->comp_max.as<uint32_t>());
    }
    if (mode != 2)
        LAUNCH(h, k_node_keep, grid_for(N + 1, 256), 256, h->node_cov.as<uint32_t>(), h->node_comp.as<uint32_t>(),
               h->comp_max.as<uint32_t>(), N, thr_node, mode, keep_n);
    if (mode != 0 && E > 0) {
        AMIRA_CUDA(cudaMemsetAsync(h->d_status.p, 0, sizeof(int) * ST_COUNT, st));
        LAUNCH(h, k_multi_edge_check, grid_for(N, 256), 256, h->e_src.as<int32_t>(), h->e_tgt.as<int32_t>(),
               h->adj_edges.as<uint32_t>(), h->adj_off.as<int64_t>(), keep_n, N, h->d_status.as<int>());
        AMIRA_CUDA(cudaMemcpyAsync(h->h_status, h->d_status.p, sizeof(int) * ST_COUNT, cudaMemcpyDeviceToHost, st));
        AMIRA_CUDA(cudaStreamSynchronize(st));
        if (h->h_status[ST_ERR] == AMIRA_E_MULTI_EDGE) {
            h->filt_N = h->filt_E = -1;  // the graph is unchanged, and keep_n no longer holds the last filter's flags
            set_error("unhashable type: 'list'");
            return AMIRA_E_MULTI_EDGE;
        }
    }
    LAUNCH(h, k_edge_keep, grid_for(E + 1, 256), 256, h->e_src.as<int32_t>(), h->e_tgt.as<int32_t>(),
           h->e_cov.as<uint32_t>(), keep_n, E, thr_edge, keep_e);
    // new indices; the sizes of the filtered graph stay on the device
    AMIRA_TRY(run_scan(h, KeepLoad{keep_n}, KeepStore{new_n, N, dsz(h, SZ_NODES)}, nullptr, 1, N, N));
    AMIRA_TRY(run_scan(h, KeepLoad{keep_e}, KeepStore{new_e, E, dsz(h, SZ_EDGES)}, nullptr, 1, E, E));
    LAUNCH(h, k_compact_nodes, grid_for(N, 256), 256, keep_n, new_n, N, k, h->node_key.as<int32_t>(),
           h->node_cov.as<uint32_t>(), h->node_dir.as<int8_t>(), h->node_comp.as<uint32_t>(), h->reads_off.as<int64_t>(),
           h->node_key2.as<int32_t>(), h->node_cov2.as<uint32_t>(), h->node_dir2.as<int8_t>(),
           h->node_comp2.as<uint32_t>(), h->reads_off2.as<int64_t>());
    // read counts of the survivors -> offsets (in place), over the new node count
    AMIRA_TRY(run_scan(h, CountLoad{h->reads_off2.as<int64_t>()},
                       OffStore{h->reads_off2.as<int64_t>(), dcnt(h, SZ_NODES), dsz(h, SZ_INC)}, dsz(h, SZ_NODES), 1, 0, N));
    LAUNCH(h, k_compact_incidence, grid_for(N * 32, 256), 256, keep_n, new_n, N, h->reads_off.as<int64_t>(),
           h->reads.as<uint32_t>(), h->reads_off2.as<int64_t>(), h->reads2.as<uint32_t>());
    if (E > 0) {
        LAUNCH(h, k_compact_edges, grid_for(E, 256), 256, keep_e, new_e, new_n, E, h->e_src.as<int32_t>(),
               h->e_tgt.as<int32_t>(), h->e_sd.as<int8_t>(), h->e_td.as<int8_t>(), h->e_cov.as<uint32_t>(),
               h->e_src2.as<int32_t>(), h->e_tgt2.as<int32_t>(), h->e_sd2.as<int8_t>(), h->e_td2.as<int8_t>(),
               h->e_cov2.as<uint32_t>());
    }
    if (W > 0) {
        LAUNCH(h, k_mask_windows, (int)std::min<int64_t>(grid_for(W, 256), (int64_t)h->n_sm * 32), 256, keep_n, new_n,
               h->win_node.as<int32_t>(), h->win_dir.as<int8_t>(), h->win_read.as<int32_t>(), (int32_t)h->first_read_global,
               h->has_pos ? h->win_start.as<int32_t>() : nullptr, h->has_pos ? h->win_end.as<int32_t>() : nullptr,
               (long long)W, h->to_correct.as<uint8_t>());
    }
    AMIRA_CUDA(cudaEventRecord(h->ev_reads_ready, h->stream));
    std::swap(h->node_key, h->node_key2);
    std::swap(h->node_cov, h->node_cov2);
    std::swap(h->node_dir, h->node_dir2);
    std::swap(h->node_comp, h->node_comp2);
    std::swap(h->reads_off, h->reads_off2);
    std::swap(h->reads, h->reads2);
    if (E > 0) {
        std::swap(h->e_src, h->e_src2);
        std::swap(h->e_tgt, h->e_tgt2);
        std::swap(h->e_sd, h->e_sd2);
        std::swap(h->e_td, h->e_td2);
        std::swap(h->e_cov, h->e_cov2);
    }
    buffer_generation()++;  // a build captured before this filter would write into the old buffers
    AMIRA_TRY(build_adjacency(h, false));
    AMIRA_TRY(enqueue_report(h, 1));
    h->pending = 2;
    h->pending_is_build = false;
    return AMIRA_OK;
}

// the status a filter / removal leaves for the calls after it.  One refused for a multi-edge changed nothing, so the
// graph stays usable and keeps the status it had (upstream's graph also survives the TypeError).
int filter_status(amira_gmg *h, int rc) {
    if (rc != AMIRA_E_MULTI_EDGE) h->last_status = rc;
    return rc;
}

// ---- multi-GPU: merge the local tables of all ranks into the global node / edge arrays ----------
// (see sharded.cuh for the scheme)
// perm[rank by first global call position] = record, for n merged records (sharded.cuh: bitmap + prefix popcount)
template <class Pos>
int rank_by_position(amira_gmg *h, const Pos pos, long long n, unsigned int *perm) {
    if (n <= 0) return AMIRA_OK;
    const int64_t n_words = h->calls_global / 32 + 1;
    AMIRA_TRY(h->x_bm.reserve(sizeof(unsigned int) * (size_t)(n_words + 1)));
    AMIRA_TRY(h->x_pref.reserve(sizeof(int) * (size_t)(n_words + 2)));
    AMIRA_CUDA(cudaMemsetAsync(h->x_bm.p, 0, sizeof(unsigned int) * (size_t)(n_words + 1), h->cur));
    h->lib_launches++;
    LAUNCH(h, k_mark_ord<Pos>, grid_for(n, 256), 256, pos, n, h->x_bm.as<unsigned int>());
    AMIRA_TRY(run_scan(h, BmLoad{h->x_bm.as<unsigned int>()}, BmStore{h->x_pref.as<int>()}, nullptr, 1, n_words, n_words));
    LAUNCH(h, k_rank_ord<Pos>, grid_for(n, 256), 256, pos, n, h->x_bm.as<unsigned int>(), h->x_pref.as<int>(), perm);
    return AMIRA_OK;
}

// counts[world] on the device -> the world x world matrix on the host (h_cnt[src * world + dst]);
// fills send_off / recv_off of this rank and zeroes the cursors for the scatter pass
int exchange_counts(amira_gmg *h, std::vector<int64_t> &send_off, std::vector<int64_t> &recv_off) {
    const int world = h->world, me = h->rank;
    unsigned long long *d_cnt = h->x_cnt.as<unsigned long long>();
    unsigned long long *d_mat = d_cnt + 2 * MAX_WORLD;
    AMIRA_TRY(comm_allgather(h->comm, d_cnt, d_mat, sizeof(unsigned long long) * world, h->cur));
    AMIRA_CUDA(cudaMemcpyAsync(h->h_cnt, d_mat, sizeof(unsigned long long) * world * world, cudaMemcpyDeviceToHost,
                               h->cur));
    AMIRA_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long) * MAX_WORLD, h->cur));
    AMIRA_CUDA(cudaStreamSynchronize(h->cur));
    send_off.assign(world + 1, 0);
    recv_off.assign(world + 1, 0);
    for (int p = 0; p < world; ++p) {
        send_off[p + 1] = send_off[p] + h->h_cnt[(int64_t)me * world + p];
        recv_off[p + 1] = recv_off[p] + h->h_cnt[(int64_t)p * world + me];
    }
    return AMIRA_OK;
}

// from the count matrix: records owner d receives in total, and where this rank's block starts there
void owner_layout(const amira_gmg *h, int d, int64_t &n_recv, int64_t &my_start) {
    n_recv = my_start = 0;
    for (int src = 0; src < h->world; ++src) {
        if (src == h->rank) my_start = n_recv;
        n_recv += h->h_cnt[(int64_t)src * h->world + d];
    }
}

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// one counter per rank -> offsets of the all-gather-v
int gather_counts(amira_gmg *h, std::vector<int64_t> &off) {
    const int world = h->world;
    unsigned long long *d_cnt = h->x_cnt.as<unsigned long long>();
    unsigned long long *d_mat = d_cnt + 2 * MAX_WORLD;
    AMIRA_TRY(comm_allgather(h->comm, d_cnt, d_mat, sizeof(unsigned long long), h->cur));
    AMIRA_CUDA(cudaMemcpyAsync(h->h_cnt, d_mat, sizeof(unsigned long long) * world, cudaMemcpyDeviceToHost, h->cur));
    AMIRA_CUDA(cudaMemcpyAsync(h->h_status, h->d_status.p, sizeof(int) * ST_COUNT, cudaMemcpyDeviceToHost, h->cur));
    AMIRA_CUDA(cudaStreamSynchronize(h->cur));
    off.assign(world + 1, 0);
    for (int p = 0; p < world; ++p) off[p + 1] = off[p] + h->h_cnt[p];
    return AMIRA_OK;
}

// all-gather-v of merged records: through the peer windows every rank copies its block straight into
// every other rank's window (copy engines over NVLink) and a barrier publishes them; otherwise NCCL
int publish_to_all(amira_gmg *h, bool p2p, const void *mine, int64_t n_mine, size_t elem, size_t win_off,
                   const std::vector<int64_t> &g_off, void *fallback_recv) {
    if (p2p) {
        PubDst dst;
        memset(&dst, 0, sizeof(dst));
        for (int q = 0; q < h->world; ++q) {
            const int p = (h->rank + q) % h->world;  // staggered: not every rank stores to rank 0 first
            dst.ptr[q] = (uint32_t *)((char *)comm_window(h->comm, p) + win_off + (size_t)g_off[h->rank] * elem);
        }
        const long long n_words = (long long)((size_t)n_mine * elem / 4);
        if (n_words > 0)
            LAUNCH(h, k_publish, std::min<int>(grid_for(n_words, 256), h->n_sm * 16), 256, (const uint32_t *)mine, n_words,
                   h->world, dst);
        return AMIRA_OK;
    }
    return comm_allgatherv(h->comm, mine, n_mine, fallback_recv, g_off.data(), elem, h->cur);
}

// AMIRA_SHARD_TRACE=1: per-step device times of the merge on stderr (developer aid)
struct MergeTrace {
    amira_gmg *h;
    bool on;
    std::vector<std::pair<const char *, cudaEvent_t>> marks;
    explicit MergeTrace(amira_gmg *h_) : h(h_), on(getenv("AMIRA_SHARD_TRACE") != nullptr) { mark("start"); }
    void mark(const char *name) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, h->cur);
        marks.push_back({name, e});
    }
    ~MergeTrace() {
        if (!on) return;
        cudaStreamSynchronize(h->cur);
        std::string line = "[merge rank " + std::to_string(h->rank) + "]";
        for (size_t i = 1; i < marks.size(); ++i) {
            float ms = 0;
            cudaEventElapsedTime(&ms, marks[i - 1].second, marks[i].second);
            char buf[96];
            snprintf(buf, sizeof(buf), " %s=%.3f", marks[i].first, ms);
            line += buf;
        }
        fprintf(stderr, "%s\n", line.c_str());
        for (auto &m : marks) cudaEventDestroy(m.second);
    }
};

// node half, on the main stream: afterwards every local slot knows its global node index and the global node
// arrays are final, so the per-read passes can start while the edges are still being exchanged
int sharded_merge_nodes(amira_gmg *h) {
    Phase ph(h, AMIRA_PH_EXCHANGE);
    MergeTrace tr(h);
    const int world = h->world, k = h->k, me = h->rank;
    cudaStream_t st = h->cur;
    const int tgrid_n = std::min<int>(grid_for(h->ncap, 256), h->n_sm * 16);
    const long long call_base = h->first_call_global;
    AMIRA_TRY(h->x_cnt.reserve(sizeof(unsigned long long) * (2 * MAX_WORLD + (size_t)world * world + 8)));
    unsigned long long *d_cnt = h->x_cnt.as<unsigned long long>();
    std::vector<int64_t> send_off, recv_off, g_off;
    const size_t key_bytes = sizeof(int32_t) * (size_t)k;
    bool p2p = comm_p2p(h->comm);

    // ---- nodes: route one record per locally-unique gene-mer to its owner
    AMIRA_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long) * MAX_WORLD, st));
    NodeDst ndst;
    memset(&ndst, 0, sizeof(ndst));
    LAUNCH(h, k_node_route<false>, tgrid_n, 256, h->nview, h->ids, k, world, call_base, d_cnt, ndst);
    AMIRA_TRY(exchange_counts(h, send_off, recv_off));
    tr.mark("n_count");
    const int64_t Nl = send_off[world], Nr = recv_off[world];
    int64_t nr_max = 0, nl_sum = 0;
    for (int d = 0; d < world; ++d) {
        int64_t n, my;
        owner_layout(h, d, n, my);
        nr_max = std::max(nr_max, n);
        nl_sum += n;
    }
    // window layout (identical on every rank): [a2a keys | a2a meta | merged keys | merged meta]; the
    // merged regions are sized for the worst case (nothing merges) so the window is mapped once
    const size_t w_meta = align256(key_bytes * nr_max), w_gkey = w_meta + align256(sizeof(NodeRec) * nr_max);
    const size_t w_gmeta = w_gkey + align256(key_bytes * nl_sum), w_end = w_gmeta + align256(sizeof(NodeRec) * nl_sum);
    if (p2p) {
        AMIRA_TRY(comm_window_ensure(h->comm, w_end, st));
        p2p = comm_p2p(h->comm);
    }
    const int32_t *r_key;
    const NodeRec *r_meta;
    if (p2p) {
        for (int d = 0; d < world; ++d) {
            int64_t n, my;
            owner_layout(h, d, n, my);
            char *w = (char *)comm_window(h->comm, d);
            ndst.key[d] = (int32_t *)w;
            ndst.meta[d] = (NodeRec *)(w + w_meta);
            ndst.start[d] = my;
        }
        LAUNCH(h, k_node_route<true>, tgrid_n, 256, h->nview, h->ids, k, world, call_base, d_cnt, ndst);
        AMIRA_TRY(comm_barrier(h->comm, st));
        r_key = (const int32_t *)comm_window(h->comm, me);
        r_meta = (const NodeRec *)((const char *)comm_window(h->comm, me) + w_meta);
    } else {
        AMIRA_TRY(h->x_skey.reserve(key_bytes * std::max<int64_t>(Nl, 1)));
        AMIRA_TRY(h->x_smeta.reserve(sizeof(NodeRec) * std::max<int64_t>(Nl, 1)));
        AMIRA_TRY(h->x_rkey.reserve(key_bytes * std::max<int64_t>(Nr, 1)));
        AMIRA_TRY(h->x_rmeta.reserve(sizeof(NodeRec) * std::max<int64_t>(Nr, 1)));
        for (int d = 0; d < world; ++d) {
            ndst.key[d] = h->x_skey.as<int32_t>();
            ndst.meta[d] = h->x_smeta.as<NodeRec>();
            ndst.start[d] = send_off[d];
        }
        LAUNCH(h, k_node_route<true>, tgrid_n, 256, h->nview, h->ids, k, world, call_base, d_cnt, ndst);
        AMIRA_TRY(comm_alltoallv(h->comm, h->x_skey.p, send_off.data(), h->x_rkey.p, recv_off.data(), key_bytes, st));
        AMIRA_TRY(comm_alltoallv(h->comm, h->x_smeta.p, send_off.data(), h->x_rmeta.p, recv_off.data(), sizeof(NodeRec), st));
        r_key = h->x_rkey.as<int32_t>();
        r_meta = h->x_rmeta.as<NodeRec>();
    }
    tr.mark("n_a2a");

    // ---- owner merge: records in first-position order into a table (sum of counts, earliest record)
    int64_t mcap = std::min<int64_t>(2 * Nr + 1024, 0x7FFFFFF0ll);
    AMIRA_TRY(h->x_tab.reserve(sizeof(NodeSlot) * mcap));
    AMIRA_TRY(h->x_mkey.reserve(key_bytes * std::max<int64_t>(Nr, 1)));
    AMIRA_TRY(h->x_mmeta.reserve(sizeof(NodeRec) * std::max<int64_t>(Nr, 1)));
    AMIRA_CUDA(cudaMemsetAsync(h->x_tab.p, 0xFF, sizeof(NodeSlot) * mcap, st));
    AMIRA_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), st));
    BuildParams P;
    memset(&P, 0, sizeof(P));
    P.k = k;
    P.status = h->d_status.as<int>();
    // earliest first occurrence per merged gene-mer (x_rmeta2 doubles as that array)
    AMIRA_TRY(h->x_rmeta2.reserve(sizeof(unsigned long long) * (size_t)mcap));
    AMIRA_CUDA(cudaMemsetAsync(h->x_rmeta2.p, 0xFF, sizeof(unsigned long long) * (size_t)mcap, st));
    if (Nr > 0) {
        P.ids = r_key;
        P.ntab = h->x_tab.as<NodeSlot>();
        P.ncap = (unsigned int)mcap;
        LAUNCH(h, k_insert_records, grid_for(Nr, 256), 256, P, (long long)Nr, r_meta, h->x_rmeta2.as<unsigned long long>());
        LAUNCH(h, k_pack_merged_nodes, std::min<int>(grid_for(mcap, 256), h->n_sm * 16), 256, h->x_tab.as<NodeSlot>(),
               (unsigned int)mcap, r_key, h->x_rmeta2.as<unsigned long long>(), k, d_cnt, h->x_mkey.as<int32_t>(),
               h->x_mmeta.as<NodeRec>());
    }
    AMIRA_TRY(gather_counts(h, g_off));
    tr.mark("n_merge");
    const int64_t Nm = g_off[h->rank + 1] - g_off[h->rank], Ng = g_off[world];
    if (Ng >= 0x7FFFFFF0ll) {
        set_error("too many nodes for int32 node indices");
        return AMIRA_E_ARG;
    }
    const int32_t *g_key;
    const NodeRec *g_meta;
    if (p2p) {
        AMIRA_TRY(publish_to_all(h, true, h->x_mkey.p, Nm, key_bytes, w_gkey, g_off, nullptr));
        AMIRA_TRY(publish_to_all(h, true, h->x_mmeta.p, Nm, sizeof(NodeRec), w_gmeta, g_off, nullptr));
        AMIRA_TRY(comm_barrier(h->comm, st));
        g_key = (const int32_t *)((const char *)comm_window(h->comm, me) + w_gkey);
        g_meta = (const NodeRec *)((const char *)comm_window(h->comm, me) + w_gmeta);
    } else {
        AMIRA_TRY(h->x_gkey.reserve(key_bytes * std::max<int64_t>(Ng, 1)));
        AMIRA_TRY(h->x_gmeta.reserve(sizeof(NodeRec) * std::max<int64_t>(Ng, 1)));
        AMIRA_TRY(publish_to_all(h, false, h->x_mkey.p, Nm, key_bytes, 0, g_off, h->x_gkey.p));
        AMIRA_TRY(publish_to_all(h, false, h->x_mmeta.p, Nm, sizeof(NodeRec), 0, g_off, h->x_gmeta.p));
        g_key = h->x_gkey.as<int32_t>();
        g_meta = h->x_gmeta.as<NodeRec>();
    }
    tr.mark("n_allgather");

    // ---- global node arrays in upstream's insertion order (= first global position)
    AMIRA_TRY(reserve_graph(h, Ng, 0));
    AMIRA_TRY(h->cov_local.reserve(sizeof(uint32_t) * (Ng + 1)));
    AMIRA_CUDA(cudaMemsetAsync(h->cov_local.p, 0, sizeof(uint32_t) * (Ng + 1), st));
    if (Ng > 0) {
        AMIRA_TRY(h->x_sorti2.reserve(sizeof(unsigned int) * Ng));
        AMIRA_TRY(rank_by_position(h, NodePos{g_meta}, (long long)Ng, h->x_sorti2.as<unsigned int>()));
        LAUNCH(h, k_finalize_nodes, grid_for(Ng, 256), 256, h->x_sorti2.as<unsigned int>(), g_key, g_meta, k, (long long)Ng, h->node_key.as<int32_t>(), h->node_cov.as<uint32_t>(),
               h->node_dir.as<int8_t>(), h->link.as<uint8_t>());
        // local slots -> global node indices: probe the rank's own node table with every global gene-mer
        if (h->G > 0)
            LAUNCH(h, k_global_to_local, grid_for(Ng, 256), 256, h->local_P, h->n16 ? 1 : 0, h->nview,
                   h->node_key.as<int32_t>(), (long long)Ng, h->cov_local.as<uint32_t>());
    }

    tr.mark("n_global");
    h->n_nodes = Ng;
    h->prev_nodes = Nl;
    return AMIRA_OK;
}

// edge half, on the CURRENT stream (the second one: it runs beside the per-read passes of the main stream)
int sharded_merge_edges(amira_gmg *h) {
    Phase ph(h, AMIRA_PH_EXCHANGE_EDGES);
    MergeTrace tr(h);
    const int world = h->world, me = h->rank;
    cudaStream_t st = h->cur;
    const int tgrid_e = std::min<int>(grid_for(h->ecap, 256), h->n_sm * 16);
    const long long call_base = h->first_call_global;
    const int64_t Ng = h->n_nodes;
    unsigned long long *d_cnt = h->x_cnt.as<unsigned long long>();
    std::vector<int64_t> send_off, recv_off, g_off;
    bool p2p = comm_p2p(h->comm);
    // ---- edges: one record per locally-unique undirected adjacency, keyed on global node indices
    AMIRA_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long) * MAX_WORLD, st));
    EdgeDst edst;
    memset(&edst, 0, sizeof(edst));
    LAUNCH(h, k_edge_route<false>, tgrid_e, 256, h->eview, h->nview, world, call_base, d_cnt, edst);
    AMIRA_TRY(exchange_counts(h, send_off, recv_off));
    tr.mark("e_count");
    const int64_t El = send_off[world], Er = recv_off[world];
    int64_t er_max = 0, el_sum = 0;
    for (int d = 0; d < world; ++d) {
        int64_t n, my;
        owner_layout(h, d, n, my);
        er_max = std::max(er_max, n);
        el_sum += n;
    }
    const size_t w_gedge = align256(sizeof(EdgeSlot) * er_max), w_eend = w_gedge + align256(sizeof(EdgeSlot) * el_sum);
    if (p2p) {
        AMIRA_TRY(comm_window_ensure(h->comm, w_eend, st));
        p2p = comm_p2p(h->comm);
    }
    const EdgeSlot *r_edge;
    if (p2p) {
        for (int d = 0; d < world; ++d) {
            int64_t n, my;
            owner_layout(h, d, n, my);
            edst.rec[d] = (EdgeSlot *)comm_window(h->comm, d);
            edst.start[d] = my;
        }
        LAUNCH(h, k_edge_route<true>, tgrid_e, 256, h->eview, h->nview, world, call_base, d_cnt, edst);
        AMIRA_TRY(comm_barrier(h->comm, st));
        r_edge = (const EdgeSlot *)comm_window(h->comm, me);
    } else {
        AMIRA_TRY(h->x_sedge.reserve(sizeof(EdgeSlot) * std::max<int64_t>(El, 1)));
        AMIRA_TRY(h->x_redge.reserve(sizeof(EdgeSlot) * std::max<int64_t>(Er, 1)));
        for (int d = 0; d < world; ++d) {
            edst.rec[d] = h->x_sedge.as<EdgeSlot>();
            edst.start[d] = send_off[d];
        }
        LAUNCH(h, k_edge_route<true>, tgrid_e, 256, h->eview, h->nview, world, call_base, d_cnt, edst);
        AMIRA_TRY(comm_alltoallv(h->comm, h->x_sedge.p, send_off.data(), h->x_redge.p, recv_off.data(), sizeof(EdgeSlot), st));
        r_edge = h->x_redge.as<EdgeSlot>();
    }
    tr.mark("e_a2a");
    AMIRA_TRY(h->x_medge.reserve(sizeof(EdgeSlot) * std::max<int64_t>(Er, 1)));
    const int64_t mecap = std::min<int64_t>(2 * Er + 1024, 0x7FFFFFF0ll);
    AMIRA_TRY(h->x_etab.reserve(sizeof(EdgeSlot) * mecap));
    AMIRA_CUDA(cudaMemsetAsync(h->x_etab.p, 0xFF, sizeof(EdgeSlot) * mecap, st));
    AMIRA_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), st));
    if (Er > 0) {
        LAUNCH(h, k_merge_edges, grid_for(Er, 256), 256, r_edge, (long long)Er, h->x_etab.as<EdgeSlot>(),
               (unsigned int)mecap, h->d_status.as<int>());
        LAUNCH(h, k_pack_merged_edges, std::min<int>(grid_for(mecap, 256), h->n_sm * 16), 256, h->x_etab.as<EdgeSlot>(),
               (unsigned int)mecap, d_cnt, h->x_medge.as<EdgeSlot>());
    }
    AMIRA_TRY(gather_counts(h, g_off));
    tr.mark("e_merge");
    const int64_t Em = g_off[h->rank + 1] - g_off[h->rank], Eg = g_off[world];
    const EdgeSlot *g_edge;
    if (p2p) {
        AMIRA_TRY(publish_to_all(h, true, h->x_medge.p, Em, sizeof(EdgeSlot), w_gedge, g_off, nullptr));
        AMIRA_TRY(comm_barrier(h->comm, st));
        g_edge = (const EdgeSlot *)((const char *)comm_window(h->comm, me) + w_gedge);
    } else {
        AMIRA_TRY(h->x_gedge.reserve(sizeof(EdgeSlot) * std::max<int64_t>(Eg, 1)));
        AMIRA_TRY(publish_to_all(h, false, h->x_medge.p, Em, sizeof(EdgeSlot), 0, g_off, h->x_gedge.p));
        g_edge = h->x_gedge.as<EdgeSlot>();
    }
    tr.mark("e_allgather");
    int64_t E_dir = 0;
    AMIRA_TRY(h->x_fan.reserve(sizeof(int) * (Eg + 2)));
    if (Eg > 0) {
        AMIRA_TRY(h->x_sorti2.reserve(sizeof(unsigned int) * Eg));
        AMIRA_TRY(rank_by_position(h, EdgePos{g_edge}, (long long)Eg, h->x_sorti2.as<unsigned int>()));
        AMIRA_TRY(run_scan(h, FanLoad{h->x_sorti2.as<unsigned int>(), g_edge}, FanStore{h->x_fan.as<int>()}, nullptr, 1, Eg, Eg));
        int e_dir32 = 0;
        AMIRA_CUDA(cudaMemcpyAsync(&e_dir32, h->x_fan.as<int>() + Eg, sizeof(int), cudaMemcpyDeviceToHost, st));
        AMIRA_CUDA(cudaMemcpyAsync(h->h_status, h->d_status.p, sizeof(int) * ST_COUNT, cudaMemcpyDeviceToHost, st));
        AMIRA_CUDA(cudaStreamSynchronize(st));
        E_dir = e_dir32;
    }
    if (h->h_status[ST_ERR] || h->h_status[ST_OVERFLOW_N] || h->h_status[ST_OVERFLOW_E]) {
        set_error("internal error while merging the sharded tables (status %d/%d/%d)", h->h_status[ST_ERR],
                  h->h_status[ST_OVERFLOW_N], h->h_status[ST_OVERFLOW_E]);
        return AMIRA_E_STATE;
    }
    AMIRA_TRY(reserve_graph(h, Ng, E_dir));
    // the directed edge arrays (+ union-find) are emitted on the second stream, beside the per-read passes
    h->sh_Eg = Eg;
    h->sh_gedge = g_edge;
    tr.mark("e_global");
    h->n_edges = E_dir;
    h->prev_und_edges = El + 1;
    return AMIRA_OK;
}

__global__ void k_sub_offset(const int64_t *__restrict__ in, int64_t n, int64_t *__restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] - in[0];
}

int d2h(amira_gmg *h, void *dst, const void *src, size_t bytes) {
    if (!dst || bytes == 0) return AMIRA_OK;
    AMIRA_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->stream));
    h->lib_launches++;
    return AMIRA_OK;
}

int check_handle(const amira_gmg *h) {
    if (!h) {
        set_error("null handle");
        return AMIRA_E_ARG;
    }
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) {
        set_error("cudaSetDevice(%d): %s", h->device, cudaGetErrorString(e));
        return AMIRA_E_CUDA;
    }
    return AMIRA_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

const char *amira_last_error(void) { return g_err; }
const char *amira_version(void) { return "amira_gmg 0.1 (sm_100a)"; }

int amira_gmg_create(amira_gmg **out, int device, void *cuda_stream) {
    if (!out) return AMIRA_E_ARG;
    *out = nullptr;
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available: %s (there is no CPU fallback)", cudaGetErrorString(e));
        return AMIRA_E_CUDA;
    }
    if (device < 0 || device >= n_dev) {
        set_error("device %d out of range (%d devices)", device, n_dev);
        return AMIRA_E_ARG;
    }
    AMIRA_CUDA(cudaSetDevice(device));
    amira_gmg *h = new amira_gmg();
    h->device = device;
    if (cuda_stream) {
        h->stream = (cudaStream_t)cuda_stream;
    } else {
        AMIRA_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        h->own_stream = true;
    }
    {
        // high priority: the second stream carries many small, latency-bound kernels that should slip in
        // between the waves of the bandwidth-bound sort on the main stream
        int prio_lo = 0, prio_hi = 0;
        AMIRA_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        const bool side_low = getenv("AMIRA_SIDE_LOW") != nullptr;  // developer experiments
        AMIRA_CUDA(cudaStreamCreateWithPriority(&h->stream2, cudaStreamNonBlocking, side_low ? prio_lo : prio_hi));
    }
    AMIRA_CUDA(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    AMIRA_CUDA(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    AMIRA_CUDA(cudaStreamCreateWithFlags(&h->stream_copy, cudaStreamNonBlocking));
    AMIRA_CUDA(cudaEventCreateWithFlags(&h->ev_reads_ready, cudaEventDisableTiming));
    AMIRA_CUDA(cudaEventCreateWithFlags(&h->ev_input_free, cudaEventDisableTiming));
    for (int i = 0; i < amira_gmg::H2D_PIECES; ++i) AMIRA_CUDA(cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming));
    h->cur = h->stream;
    cudaDeviceProp prop;
    AMIRA_CUDA(cudaGetDeviceProperties(&prop, device));
    h->n_sm = prop.multiProcessorCount;
    AMIRA_CUDA(cudaFuncSetAttribute(k_unit_lists, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)INC_SMEM));
    AMIRA_CUDA(cudaFuncSetAttribute(k_union_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(int32_t) * UF_SMALL_RUNS)));
    AMIRA_CUDA(cudaFuncSetAttribute(k_partition<PartSmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PartSmall::SMEM));
    AMIRA_CUDA(cudaFuncSetAttribute(k_partition<PartWide>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PartWide::SMEM));
    AMIRA_CUDA(cudaFuncSetAttribute(k_partition<PartBig>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PartBig::SMEM));
    int occ = 1;
    AMIRA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (k_insert_windows<5, true, true>), INS_THREADS, 0));
    h->insert_ctas_per_sm = std::max(1, occ);
    AMIRA_TRY(h->d_status.reserve(sizeof(int) * ST_COUNT));
    AMIRA_TRY(h->d_sizes.reserve(sizeof(long long) * SZ_COUNT));
    AMIRA_CUDA(cudaMallocHost((void **)&h->h_status, sizeof(int) * 2 * ST_COUNT));
    AMIRA_CUDA(cudaMallocHost((void **)&h->h_sizes, sizeof(long long) * 2 * SZ_COUNT));
    AMIRA_CUDA(cudaEventCreateWithFlags(&h->ev_early, cudaEventDisableTiming));
    AMIRA_CUDA(cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming));
    AMIRA_CUDA(cudaFuncSetAttribute(k_segsort_radix, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 + 2 * 4 * SEG_STAGE_MAX));
    for (int i = 0; i < AMIRA_PH_COUNT; ++i)
        for (int j = 0; j < 2; ++j) AMIRA_CUDA(cudaEventCreate(&h->ev[i][j]));
    *out = h;
    return AMIRA_OK;
}

void amira_gmg_destroy(amira_gmg *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->stream2) {
        cudaStreamSynchronize(h->stream2);
        cudaStreamDestroy(h->stream2);
    }
    if (h->stream_copy) {
        cudaStreamSynchronize(h->stream_copy);
        cudaStreamDestroy(h->stream_copy);
    }
    if (h->ev_reads_ready) cudaEventDestroy(h->ev_reads_ready);
    if (h->ev_input_free) cudaEventDestroy(h->ev_input_free);
    for (int i = 0; i < amira_gmg::H2D_PIECES; ++i)
        if (h->ev_h2d[i]) cudaEventDestroy(h->ev_h2d[i]);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    DevBuf *bufs[] = {&h->d_ids, &h->d_off, &h->d_ps, &h->d_pe, &h->win_off, &h->is_short, &h->to_correct, &h->tile_r0,
                      &h->win_node, &h->win_dir, &h->win_read, &h->win_start, &h->win_end, &h->ntab, &h->etab,
                      &h->bitmaps, &h->cnt_node, &h->cnt_edge, &h->node_key, &h->node_cov, &h->node_dir, &h->node_comp,
                      &h->reads_off, &h->reads, &h->node_key2, &h->node_cov2, &h->node_dir2, &h->node_comp2,
                      &h->reads_off2, &h->reads2, &h->parent, &h->link, &h->run_id, &h->run_pairs, &h->is_root, &h->e_src, &h->e_tgt, &h->e_sd, &h->e_td,
                      &h->e_cov, &h->e_src2, &h->e_tgt2, &h->e_sd2, &h->e_td2, &h->e_cov2, &h->adj_off, &h->adj_edges,
                      &h->adj_cursor, &h->adj_tmp, &h->reads_tmp, &h->slot_info, &h->inc_rec, &h->unit_lo, &h->bucket_cursor, &h->win_slot, &h->seg_work[0], &h->seg_work[1], &h->scan_state[0], &h->scan_state[1], &h->scan_pool, &h->dups,
                      &h->keep_n, &h->keep_e, &h->comp_max, &h->scratch_off, &h->d_status, &h->d_sizes,
                      &h->x_cnt, &h->x_skey, &h->x_smeta, &h->x_rkey, &h->x_rmeta, &h->x_rmeta2,
                      &h->x_mkey, &h->x_mmeta, &h->x_gkey, &h->x_gmeta, &h->x_tab, &h->x_bm, &h->x_pref,
                      &h->x_sorti2, &h->x_sedge, &h->x_redge, &h->x_medge, &h->x_gedge, &h->x_etab, &h->x_fan,
                      &h->cov_local, &h->cc_min, &h->d_maxabs};
    for (DevBuf *b : bufs) b->release();
    if (h->comm) comm_destroy(h->comm);
    if (h->h_cnt) cudaFreeHost(h->h_cnt);
    if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
    if (h->ev_early) cudaEventDestroy(h->ev_early);
    if (h->ev_done) cudaEventDestroy(h->ev_done);
    if (h->h_status) cudaFreeHost(h->h_status);
    if (h->h_sizes) cudaFreeHost(h->h_sizes);
    for (int i = 0; i < AMIRA_PH_COUNT; ++i)
        for (int j = 0; j < 2; ++j)
            if (h->ev[i][j]) cudaEventDestroy(h->ev[i][j]);
    if (h->own_stream) cudaStreamDestroy(h->stream);
    delete h;
}

int amira_gmg_reserve(amira_gmg *h, int64_t n_nodes_hint, int64_t n_edges_hint) {
    AMIRA_TRY(check_handle(h));
    h->hint_nodes = n_nodes_hint;
    h->hint_edges = n_edges_hint;
    return AMIRA_OK;
}

int amira_gmg_set_profiling(amira_gmg *h, int enabled) {
    AMIRA_TRY(check_handle(h));
    h->profiling = enabled != 0;
    return AMIRA_OK;
}

int amira_gmg_phase_ms(const amira_gmg *h, int phase, float *ms) {
    if (!h || !ms || phase < 0 || phase >= AMIRA_PH_COUNT) return AMIRA_E_ARG;
    *ms = 0.f;
    if (!h->ev_used[phase]) return AMIRA_OK;
    cudaError_t e = cudaEventElapsedTime(ms, h->ev[phase][0], h->ev[phase][1]);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *ms = 0.f;
    }
    return AMIRA_OK;
}

int amira_gmg_kernel_launches(const amira_gmg *h, int64_t *n) {
    if (!h || !n) return AMIRA_E_ARG;
    *n = h->launches;
    return AMIRA_OK;
}

int amira_gmg_build(amira_gmg *h, const int32_t *signed_ids, const int64_t *read_off, int64_t R, int32_t k,
                    const int32_t *pos_start, const int32_t *pos_end, int input_on_device) {
    AMIRA_TRY(check_handle(h));
    // a previous build nobody looked at: keep what it learned (table sizes, id width) if it has finished
    if (h->pending && h->pending_is_build && h->world == 1 && cudaEventQuery(h->ev_done) == cudaSuccess) finish(h, false);
    cudaGetLastError();
    h->built = false;
    h->filt_N = h->filt_E = -1;
    reset_graph(h);
    h->attempts = 0;
    for (int i = 0; i < AMIRA_PH_COUNT; ++i) h->ev_used[i] = false;
    int arg_status = AMIRA_OK;
    if (R < 0 || k < 0 || (R > 0 && !read_off) || ((pos_start == nullptr) != (pos_end == nullptr))) {
        set_error("bad arguments to amira_gmg_build");
        arg_status = AMIRA_E_ARG;
    } else if (R >= 0x7FFFFFF0ll) {
        set_error("too many reads for int32 read indices");
        arg_status = AMIRA_E_ARG;
    } else if (k > MAX_K) {
        set_error("k=%d exceeds the supported maximum %d", k, MAX_K);
        arg_status = AMIRA_E_ARG;
    } else if (k == 0 && (R > 0 || h->world > 1)) {  // GeneMer([]) for every read: "Gene-mer is empty"
        set_error("Gene-mer is empty");
        arg_status = AMIRA_E_EMPTY_GENEMER;
    }
    cudaStream_t st = h->stream;
    int64_t G = 0;
    h->input_on_device = input_on_device != 0;
    if (arg_status == AMIRA_OK && R > 0) {
        if (input_on_device) {
            if (read_off == h->cache_off && R == h->cache_R) {
                G = h->cache_G;  // verified on the device by the per-read pass (ST_STALE)
            } else {
                AMIRA_CUDA(cudaMemcpyAsync(&G, read_off + R, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
                AMIRA_CUDA(cudaStreamSynchronize(st));
                h->cache_off = read_off;
                h->cache_R = R;
                h->cache_G = G;
            }
        } else {
            G = read_off[R];
        }
        if (G < 0 || G >= MAX_CALLS || (G > 0 && !signed_ids)) {
            set_error("bad call count %lld", (long long)G);
            h->cache_off = nullptr;
            arg_status = AMIRA_E_ARG;
        }
    }
    if (h->world > 1) {
        // collective build: every rank must take the same exit, so the argument status is agreed first
        AMIRA_TRY(h->x_cnt.reserve(sizeof(unsigned long long) * (2 * MAX_WORLD + (size_t)h->world * h->world + 8)));
        int *d_arg = h->x_cnt.as<int>();
        AMIRA_CUDA(cudaMemcpyAsync(d_arg, &arg_status, sizeof(int), cudaMemcpyHostToDevice, h->stream));
        AMIRA_TRY(comm_allreduce_max_i32(h->comm, d_arg, 1, h->stream));
        int agreed = 0;
        AMIRA_CUDA(cudaMemcpyAsync(&agreed, d_arg, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        AMIRA_CUDA(cudaStreamSynchronize(h->stream));
        if (agreed != AMIRA_OK && arg_status == AMIRA_OK) {
            set_error("another rank rejected its arguments to the collective amira_gmg_build (status %d)", agreed);
            arg_status = agreed;
        }
    }
    if (arg_status != AMIRA_OK) return h->last_status = arg_status;
    h->R = R;
    h->k = k;
    h->has_pos = pos_start != nullptr;
    h->G = 0;
    h->last_status = AMIRA_OK;
    if (R == 0 && h->world == 1) {  // GeneMerGraph({}, k): empty graph for any k (tests/test_gene_mer_graph.py:14-36)
        h->built = true;
        return AMIRA_OK;
    }
    h->G = G;
    h->n_pieces = 0;
    bool wait_h2d = false;
    if (input_on_device) {
        h->ids = signed_ids;
        h->off = read_off;
        h->ps = pos_start;
        h->pe = pos_end;
    } else {
        Phase ph(h, AMIRA_PH_H2D);
        AMIRA_TRY(h->d_ids.reserve(sizeof(int32_t) * std::max<int64_t>(G, 1) + 16));
        AMIRA_TRY(h->d_off.reserve(sizeof(int64_t) * (R + 1)));
        // offsets first (the per-read pass needs only them), then the ids in pieces on the copy stream
        if (read_off) AMIRA_CUDA(cudaMemcpyAsync(h->d_off.p, read_off, sizeof(int64_t) * (R + 1), cudaMemcpyHostToDevice, st));
        else AMIRA_CUDA(cudaMemsetAsync(h->d_off.p, 0, sizeof(int64_t) * (R + 1), st));
        if (G >= (int64_t)amira_gmg::H2D_PIECES * (1 << 20) && !h->has_pos) {
            AMIRA_CUDA(cudaEventRecord(h->ev_input_free, st));  // earlier work on the main stream may still read d_ids
            AMIRA_CUDA(cudaStreamWaitEvent(h->stream_copy, h->ev_input_free, 0));
            int64_t begin = 0;
            for (int i = 0; i < amira_gmg::H2D_PIECES; ++i) {
                int64_t end = (i + 1 == amira_gmg::H2D_PIECES) ? G : ((G * (i + 1) / amira_gmg::H2D_PIECES) / INS_TILE) * INS_TILE;
                AMIRA_CUDA(cudaMemcpyAsync(h->d_ids.as<int32_t>() + begin, signed_ids + begin, sizeof(int32_t) * (end - begin),
                                           cudaMemcpyHostToDevice, h->stream_copy));
                AMIRA_CUDA(cudaEventRecord(h->ev_h2d[i], h->stream_copy));
                h->piece_end[i] = end;
                begin = end;
            }
            h->n_pieces = amira_gmg::H2D_PIECES;
        } else if (G > 0) {
            AMIRA_CUDA(cudaMemcpyAsync(h->d_ids.p, signed_ids, sizeof(int32_t) * G, cudaMemcpyHostToDevice, st));
        }
        h->ids = h->d_ids.as<int32_t>();
        h->off = h->d_off.as<int64_t>();
        h->ps = h->pe = nullptr;
        if (h->has_pos) {
            AMIRA_TRY(h->d_ps.reserve(sizeof(int32_t) * std::max<int64_t>(G, 1)));
            AMIRA_TRY(h->d_pe.reserve(sizeof(int32_t) * std::max<int64_t>(G, 1)));
            if (G > 0) {
                AMIRA_CUDA(cudaMemcpyAsync(h->d_ps.p, pos_start, sizeof(int32_t) * G, cudaMemcpyHostToDevice, st));
                AMIRA_CUDA(cudaMemcpyAsync(h->d_pe.p, pos_end, sizeof(int32_t) * G, cudaMemcpyHostToDevice, st));
            }
            h->ps = h->d_ps.as<int32_t>();
            h->pe = h->d_pe.as<int32_t>();
        }
        AMIRA_CUDA(cudaEventRecord(h->ev_input_free, st));  // the caller's buffers are free again after this point
        wait_h2d = true;
        h->lib_launches += 2;
    }
    h->first_read_global = h->first_call_global = 0;
    if (h->world > 1) {
        // contiguous shards in rank order: this rank's first global read / call index
        long long mine[2] = {(long long)R, (long long)G};
        unsigned long long *d_cnt = h->x_cnt.as<unsigned long long>();
        AMIRA_CUDA(cudaMemcpyAsync(d_cnt, mine, sizeof(mine), cudaMemcpyHostToDevice, st));
        AMIRA_TRY(comm_allgather(h->comm, d_cnt, d_cnt + 2 * MAX_WORLD, sizeof(mine), st));
        AMIRA_CUDA(cudaMemcpyAsync(h->h_cnt, d_cnt + 2 * MAX_WORLD, sizeof(mine) * h->world, cudaMemcpyDeviceToHost, st));
        AMIRA_CUDA(cudaStreamSynchronize(st));
        long long r_all = 0, g_all = 0;
        bool bad = false;
        for (int p = 0; p < h->world; ++p) {
            if (p == h->rank) {
                h->first_read_global = r_all;
                h->first_call_global = g_all;
            }
            bad |= h->h_cnt[2 * p + 1] < 0 || h->h_cnt[2 * p + 1] >= (1ll << (P_BITS - 1));
            r_all += h->h_cnt[2 * p];
            g_all += h->h_cnt[2 * p + 1];
        }
        h->calls_global = g_all;
        if (bad || r_all >= 0x7FFFFFF0ll || g_all >= (1ll << (P_BITS - 1))) {  // the same verdict on every rank
            set_error("global read set too large or inconsistent (%lld reads, %lld calls)", r_all, g_all);
            return h->last_status = AMIRA_E_ARG;
        }
        if (!h->off) {  // an empty shard still needs a valid offsets array
            AMIRA_TRY(h->d_off.reserve(sizeof(int64_t) * 2));
            AMIRA_CUDA(cudaMemsetAsync(h->d_off.p, 0, sizeof(int64_t) * 2, st));
            h->off = h->d_off.as<int64_t>();
        }
    }
    int rc = do_build(h);
    if (wait_h2d && rc == AMIRA_OK) {
        // host input: the caller may reuse its buffers as soon as this call returns
        if (h->n_pieces) AMIRA_CUDA(cudaEventSynchronize(h->ev_h2d[h->n_pieces - 1]));
        AMIRA_CUDA(cudaEventSynchronize(h->ev_input_free));
    }
    h->last_status = rc;
    h->built = (rc == AMIRA_OK);
    return rc;
}

int amira_gmg_sync(amira_gmg *h) {
    AMIRA_TRY(check_handle(h));
    const int rc = finish(h, false);
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    return rc != AMIRA_OK ? rc : h->last_status;
}

int amira_gmg_sizes(amira_gmg *h, int64_t *n_nodes, int64_t *n_edges, int64_t *n_windows, int64_t *n_incidence,
                    int64_t *n_fw, int64_t *n_bw, int64_t *n_short) {
    AMIRA_TRY(check_handle(h));
    if (!h->built) {
        set_error("sizes before a successful build");
        return AMIRA_E_STATE;
    }
    // incidence / adjacency sizes are only known when the whole build has finished; the others earlier
    AMIRA_TRY(finish(h, !(n_incidence || n_fw || n_bw)));
    if (!h->built) return h->last_status;
    if (n_nodes) *n_nodes = h->n_nodes;
    if (n_edges) *n_edges = h->n_edges;
    if (n_windows) *n_windows = h->W;
    if (n_incidence) *n_incidence = h->n_inc;
    if (n_fw) *n_fw = h->n_fw;
    if (n_bw) *n_bw = h->n_bw;
    if (n_short) *n_short = h->n_short;
    return AMIRA_OK;
}

int amira_gmg_export_nodes(amira_gmg *h, int32_t *key, uint32_t *cov, int8_t *first_dir, uint32_t *component,
                           int64_t *reads_off, int32_t *reads, int64_t *fw_off, int32_t *fw_edges, int64_t *bw_off,
                           int32_t *bw_edges) {
    AMIRA_TRY(check_handle(h));
    if (!h->built) {
        set_error("export before a successful build");
        return AMIRA_E_STATE;
    }
    AMIRA_TRY(finish(h, false));
    if (!h->built) return h->last_status;
    const int64_t N = h->n_nodes;
    if (N == 0) {
        if (reads_off) reads_off[0] = 0;
        if (fw_off) fw_off[0] = 0;
        if (bw_off) bw_off[0] = 0;
        return AMIRA_OK;
    }
    AMIRA_TRY(d2h(h, key, h->node_key.p, sizeof(int32_t) * N * h->k));
    AMIRA_TRY(d2h(h, cov, h->node_cov.p, sizeof(uint32_t) * N));
    AMIRA_TRY(d2h(h, first_dir, h->node_dir.p, N));
    AMIRA_TRY(d2h(h, component, h->node_comp.p, sizeof(uint32_t) * N));
    AMIRA_TRY(d2h(h, reads_off, h->reads_off.p, sizeof(int64_t) * (N + 1)));
    AMIRA_TRY(d2h(h, reads, h->reads.p, sizeof(int32_t) * h->n_inc));
    AMIRA_TRY(d2h(h, fw_off, h->adj_off.p, sizeof(int64_t) * (N + 1)));
    AMIRA_TRY(d2h(h, fw_edges, h->adj_edges.p, sizeof(int32_t) * h->n_fw));
    if (bw_off) {
        AMIRA_TRY(h->scratch_off.reserve(sizeof(int64_t) * (N + 1)));
        LAUNCH(h, k_sub_offset, grid_for(N + 1, 256), 256, h->adj_off.as<int64_t>() + N, N + 1,
               h->scratch_off.as<int64_t>());
        AMIRA_TRY(d2h(h, bw_off, h->scratch_off.p, sizeof(int64_t) * (N + 1)));
    }
    AMIRA_TRY(d2h(h, bw_edges, h->adj_edges.as<int32_t>() + h->n_fw, sizeof(int32_t) * h->n_bw));
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    return AMIRA_OK;
}

int amira_gmg_export_edges(amira_gmg *h, int32_t *src, int32_t *tgt, int8_t *sd, int8_t *td, uint32_t *cov) {
    AMIRA_TRY(check_handle(h));
    if (!h->built) {
        set_error("export before a successful build");
        return AMIRA_E_STATE;
    }
    AMIRA_TRY(finish(h, false));
    if (!h->built) return h->last_status;
    const int64_t E = h->n_edges;
    if (E == 0) return AMIRA_OK;
    AMIRA_TRY(d2h(h, src, h->e_src.p, sizeof(int32_t) * E));
    AMIRA_TRY(d2h(h, tgt, h->e_tgt.p, sizeof(int32_t) * E));
    AMIRA_TRY(d2h(h, sd, h->e_sd.p, E));
    AMIRA_TRY(d2h(h, td, h->e_td.p, E));
    AMIRA_TRY(d2h(h, cov, h->e_cov.p, sizeof(uint32_t) * E));
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    return AMIRA_OK;
}

int amira_gmg_export_reads(amira_gmg *h, int64_t *win_off, int32_t *node_idx, int8_t *dir, int32_t *start,
                           int32_t *end, uint8_t *is_short, uint8_t *to_correct) {
    AMIRA_TRY(check_handle(h));
    if (!h->built) {
        set_error("export before a successful build");
        return AMIRA_E_STATE;
    }
    if (h->R == 0) {
        if (win_off) win_off[0] = 0;
        return AMIRA_OK;
    }
    if ((start || end) && !h->has_pos) {
        set_error("positions requested but none were supplied to the build");
        return AMIRA_E_STATE;
    }
    AMIRA_TRY(finish(h, true));
    if (!h->built) return h->last_status;
    const int64_t W = h->W, R = h->R;
    // the per-read lists are final before the rest of the build is: copy them out beside it
    cudaStream_t cs = h->stream_copy;
    AMIRA_CUDA(cudaStreamWaitEvent(cs, h->ev_reads_ready, 0));
    struct {
        void *dst;
        const void *src;
        size_t bytes;
    } jobs[] = {{win_off, h->win_off.p, sizeof(int64_t) * (size_t)(R + 1)}, {node_idx, h->win_node.p, sizeof(int32_t) * (size_t)W},
                {dir, h->win_dir.p, (size_t)W}, {start, h->win_start.p, sizeof(int32_t) * (size_t)W},
                {end, h->win_end.p, sizeof(int32_t) * (size_t)W}, {is_short, h->is_short.p, (size_t)R},
                {to_correct, h->to_correct.p, (size_t)R}};
    for (auto &j : jobs) {
        if (!j.dst || j.bytes == 0) continue;
        AMIRA_CUDA(cudaMemcpyAsync(j.dst, j.src, j.bytes, cudaMemcpyDeviceToHost, cs));
        h->lib_launches++;
    }
    AMIRA_CUDA(cudaStreamSynchronize(cs));
    return AMIRA_OK;
}

int amira_gmg_remove_low_coverage_components(amira_gmg *h, uint32_t min_component_cov) {
    AMIRA_TRY(check_handle(h));
    return filter_status(h, do_filter(h, 1, min_component_cov, 0));
}

int amira_gmg_filter(amira_gmg *h, uint32_t min_node_cov, uint32_t min_edge_cov) {
    AMIRA_TRY(check_handle(h));
    return filter_status(h, do_filter(h, 0, min_node_cov, min_edge_cov));
}

int amira_gmg_filter_mask_sizes(amira_gmg *h, int64_t *n_nodes_before, int64_t *n_edges_before) {
    AMIRA_TRY(check_handle(h));
    if (!h->built || h->filt_N < 0) {
        set_error("no filter has run on this graph");
        return AMIRA_E_STATE;
    }
    if (n_nodes_before) *n_nodes_before = h->filt_N;
    if (n_edges_before) *n_edges_before = h->filt_E;
    return AMIRA_OK;
}

int amira_gmg_export_filter_masks(amira_gmg *h, int32_t *node_keep, int32_t *edge_keep) {
    AMIRA_TRY(check_handle(h));
    if (!h->built || h->filt_N < 0) {
        set_error("no filter has run on this graph");
        return AMIRA_E_STATE;
    }
    if (h->filt_N == 0) return AMIRA_OK;
    AMIRA_TRY(finish(h, false));
    AMIRA_TRY(d2h(h, node_keep, h->keep_n.p, sizeof(int) * h->filt_N));
    AMIRA_TRY(d2h(h, edge_keep, h->keep_e.p, sizeof(int) * h->filt_E));
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    return AMIRA_OK;
}

int amira_gmg_debug_layout(amira_gmg *h, int mask) {
    AMIRA_TRY(check_handle(h));
    h->force_layout = mask;
    return AMIRA_OK;
}

// ---- post-build scans (stats.cuh) ---------------------------------------------------------------------
namespace {
int stats_ready(amira_gmg *h) {
    AMIRA_TRY(check_handle(h));
    if (!h->built) {
        set_error("no graph on this handle");
        return AMIRA_E_STATE;
    }
    AMIRA_TRY(finish(h, false));
    return h->built ? AMIRA_OK : h->last_status;
}
}  // namespace

int amira_gmg_read_length_coverages(amira_gmg *h, const int32_t *min_len, int32_t n, int64_t *sums) {
    AMIRA_TRY(stats_ready(h));
    if (n < 0 || n > STAT_MAX_THRESHOLDS || (n > 0 && (!min_len || !sums))) {
        set_error("at most %d thresholds", STAT_MAX_THRESHOLDS);
        return AMIRA_E_ARG;
    }
    Thresholds T;
    T.n = n;
    for (int i = 0; i < n; ++i) T.min_len[i] = min_len[i];
    AMIRA_TRY(h->comp_max.reserve(sizeof(unsigned long long) * STAT_MAX_THRESHOLDS));
    unsigned long long *d_sums = h->comp_max.as<unsigned long long>();
    AMIRA_CUDA(cudaMemsetAsync(d_sums, 0, sizeof(unsigned long long) * STAT_MAX_THRESHOLDS, h->stream));
    if (h->n_inc > 0 && n > 0)
        LAUNCH(h, k_read_length_coverages, (int)std::min<int64_t>(grid_for(h->n_inc, 256), (int64_t)h->n_sm * 16), 256,
               h->reads_off.as<int64_t>(), h->reads.as<uint32_t>(), h->off, (long long)h->n_inc, (int32_t)h->first_read_global, T,
               d_sums);
    unsigned long long out[STAT_MAX_THRESHOLDS];
    AMIRA_CUDA(cudaMemcpyAsync(out, d_sums, sizeof(out), cudaMemcpyDeviceToHost, h->stream));
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n; ++i) sums[i] = (int64_t)out[i];
    return AMIRA_OK;
}

int amira_gmg_node_coverage_stats(amira_gmg *h, int64_t *sum_cov, uint32_t *max_cov) {
    AMIRA_TRY(stats_ready(h));
    AMIRA_TRY(h->comp_max.reserve(sizeof(unsigned long long) * STAT_MAX_THRESHOLDS));
    unsigned long long *d = h->comp_max.as<unsigned long long>();
    AMIRA_CUDA(cudaMemsetAsync(d, 0, sizeof(unsigned long long) * 2, h->stream));
    if (h->n_nodes > 0)
        LAUNCH(h, k_coverage_sum, (int)std::min<int64_t>(grid_for(h->n_nodes, 256), (int64_t)h->n_sm * 8), 256,
               h->node_cov.as<uint32_t>(), (long long)h->n_nodes, d);
    unsigned long long out[2];
    AMIRA_CUDA(cudaMemcpyAsync(out, d, sizeof(out), cudaMemcpyDeviceToHost, h->stream));
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    if (sum_cov) *sum_cov = (int64_t)out[0];
    if (max_cov) *max_cov = (uint32_t)out[1];
    return AMIRA_OK;
}

int amira_gmg_junk_read_mask(amira_gmg *h, double error_rate, uint8_t *mask) {
    AMIRA_TRY(stats_ready(h));
    if (h->R == 0) return AMIRA_OK;
    if (!mask) {
        set_error("junk_read_mask: no output buffer");
        return AMIRA_E_ARG;
    }
    AMIRA_TRY(h->scratch_off.reserve((size_t)h->R + 8));
    LAUNCH(h, k_junk_read_mask, grid_for(h->R, 256), 256, h->win_off.as<int64_t>(), h->win_node.as<int32_t>(),
           h->is_short.as<uint8_t>(), (long long)h->R, error_rate, h->scratch_off.as<uint8_t>());
    AMIRA_CUDA(cudaMemcpyAsync(mask, h->scratch_off.p, (size_t)h->R, cudaMemcpyDeviceToHost, h->stream));
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    return AMIRA_OK;
}

namespace {
// flags[i] = node i holds one of the genes; left on the device in scratch_off (N bytes), ranks in comp_max
int flag_nodes_containing(amira_gmg *h, const int32_t *ranks, int32_t n) {
    if (n < 0 || (n > 0 && !ranks)) {
        set_error("bad gene ranks (n = %d)", n);
        return AMIRA_E_ARG;
    }
    const int64_t N = h->n_nodes;
    AMIRA_TRY(h->scratch_off.reserve((size_t)std::max<int64_t>(N, h->R) + 8));
    AMIRA_TRY(h->comp_max.reserve(sizeof(int32_t) * (size_t)std::max(n, 1) + sizeof(uint32_t) * (size_t)(h->n_comps + 2)));
    if (n > 0) AMIRA_CUDA(cudaMemcpyAsync(h->comp_max.p, ranks, sizeof(int32_t) * n, cudaMemcpyHostToDevice, h->stream));
    if (N > 0)
        LAUNCH(h, k_nodes_containing, grid_for(N, 256), 256, h->node_key.as<int32_t>(), (long long)N, h->k, h->comp_max.as<int32_t>(),
               n, h->scratch_off.as<uint8_t>());
    return AMIRA_OK;
}
}  // namespace

int amira_gmg_nodes_containing(amira_gmg *h, const int32_t *ranks, int32_t n, uint8_t *flags) {
    AMIRA_TRY(stats_ready(h));
    AMIRA_TRY(flag_nodes_containing(h, ranks, n));
    if (h->n_nodes > 0) {
        if (!flags) return AMIRA_E_ARG;
        AMIRA_CUDA(cudaMemcpyAsync(flags, h->scratch_off.p, (size_t)h->n_nodes, cudaMemcpyDeviceToHost, h->stream));
    }
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    return AMIRA_OK;
}

int amira_gmg_remove_nodes(amira_gmg *h, const uint8_t *remove_flags) {
    AMIRA_TRY(check_handle(h));
    AMIRA_TRY(filter_reserve(h));
    const int64_t N = h->n_nodes;
    // an empty graph still goes through do_filter: the filter masks must then describe this call (zero nodes),
    // not the previous one
    if (N > 0) {
        if (!remove_flags) {
            set_error("remove_nodes: no flags for %lld nodes", (long long)N);
            return AMIRA_E_ARG;
        }
        std::vector<int> keep((size_t)N + 1);
        for (int64_t i = 0; i < N; ++i) keep[i] = remove_flags[i] ? 0 : 1;
        keep[N] = 0;
        AMIRA_CUDA(cudaMemcpyAsync(h->keep_n.p, keep.data(), sizeof(int) * (N + 1), cudaMemcpyHostToDevice, h->stream));
        AMIRA_CUDA(cudaStreamSynchronize(h->stream));  // `keep` goes out of scope
    }
    return filter_status(h, do_filter(h, 2, 0, 0));
}

int amira_gmg_remove_nodes_without_reads_of(amira_gmg *h, const int32_t *ranks, int32_t n) {
    AMIRA_TRY(check_handle(h));
    AMIRA_TRY(filter_reserve(h));
    const int64_t N = h->n_nodes, R = h->R;
    if (N == 0) return filter_status(h, do_filter(h, 2, 0, 0));  // as in amira_gmg_remove_nodes
    AMIRA_TRY(flag_nodes_containing(h, ranks, n));
    // reads of the flagged nodes (byte flags behind the node flags), then the nodes that touch none of them
    AMIRA_TRY(h->dups.reserve((size_t)R + 8));
    uint8_t *read_flag = h->dups.as<uint8_t>();
    AMIRA_CUDA(cudaMemsetAsync(read_flag, 0, (size_t)R + 1, h->stream));
    LAUNCH(h, k_mark_reads_of_nodes, grid_for(N * 32, 256), 256, h->scratch_off.as<uint8_t>(), h->reads_off.as<int64_t>(),
           h->reads.as<uint32_t>(), (long long)N, (int32_t)h->first_read_global, read_flag);
    LAUNCH(h, k_nodes_with_marked_reads, grid_for((N + 1) * 32, 256), 256, read_flag, h->reads_off.as<int64_t>(),
           h->reads.as<uint32_t>(), (long long)N, (int32_t)h->first_read_global, h->keep_n.as<int>());
    return filter_status(h, do_filter(h, 2, 0, 0));
}

int amira_gmg_linear_steps(amira_gmg *h, uint32_t *degree, int32_t *fw_next, int8_t *fw_dir, uint8_t *fw_ext, int32_t *bw_next,
                           int8_t *bw_dir, uint8_t *bw_ext) {
    AMIRA_TRY(stats_ready(h));
    const int64_t N = h->n_nodes;
    h->filt_N = h->filt_E = -1;  // the steps are computed in keep_e, the edge mask of the last filter
    if (N == 0) return AMIRA_OK;
    // [degree u32][next fw i32][next bw i32][dir fw i8][dir bw i8][ext fw u8][ext bw u8] per node
    AMIRA_TRY(h->keep_e.reserve((size_t)N * 16 + 64));
    char *base = h->keep_e.as<char>();
    LinearSteps S;
    S.degree = (uint32_t *)base;
    S.next[0] = (int32_t *)(base + 4 * N);
    S.next[1] = (int32_t *)(base + 8 * N);
    S.dir[0] = (int8_t *)(base + 12 * N);
    S.dir[1] = (int8_t *)(base + 13 * N);
    S.ext[0] = (uint8_t *)(base + 14 * N);
    S.ext[1] = (uint8_t *)(base + 15 * N);
    LAUNCH(h, k_linear_steps, grid_for(N, 256), 256, h->adj_off.as<int64_t>(), h->adj_edges.as<uint32_t>(), h->e_tgt.as<int32_t>(),
           h->e_td.as<int8_t>(), (long long)N, S);
    AMIRA_TRY(d2h(h, degree, S.degree, sizeof(uint32_t) * N));
    AMIRA_TRY(d2h(h, fw_next, S.next[0], sizeof(int32_t) * N));
    AMIRA_TRY(d2h(h, bw_next, S.next[1], sizeof(int32_t) * N));
    AMIRA_TRY(d2h(h, fw_dir, S.dir[0], N));
    AMIRA_TRY(d2h(h, bw_dir, S.dir[1], N));
    AMIRA_TRY(d2h(h, fw_ext, S.ext[0], N));
    AMIRA_TRY(d2h(h, bw_ext, S.ext[1], N));
    AMIRA_CUDA(cudaStreamSynchronize(h->stream));
    return AMIRA_OK;
}

int amira_gmg_debug_segsort(amira_gmg *h, uint32_t *data, const int64_t *off, int64_t n_seg, uint32_t *dups,
                            int64_t *total_dups, int out_of_place, int64_t max_value) {
    AMIRA_TRY(check_handle(h));
    if (!data || !off || n_seg < 0) return AMIRA_E_ARG;
    AMIRA_TRY(finish(h, false));
    const int64_t n = off[n_seg];
    DevBuf d_a, d_b, d_off, d_dups, d_cnt, d_start;
    AMIRA_TRY(d_a.reserve(sizeof(uint32_t) * std::max<int64_t>(n, 1)));
    AMIRA_TRY(d_b.reserve(sizeof(uint32_t) * std::max<int64_t>(n, 1)));
    AMIRA_TRY(d_off.reserve(sizeof(int64_t) * (n_seg + 1)));
    AMIRA_TRY(d_dups.reserve(sizeof(uint32_t) * (n_seg + 1)));
    AMIRA_TRY(d_start.reserve(sizeof(uint32_t) * (n_seg + 1)));
    AMIRA_TRY(d_cnt.reserve(2 * sizeof(long long)));
    long long cnt[2] = {(long long)n_seg, 0};
    cudaStream_t st = h->stream;
    std::vector<uint32_t> src(std::max<int64_t>(n, 1)), start(n_seg + 1);
    if (out_of_place) {
        // the source holds the segments in REVERSE order: exercises a_start
        int64_t pos = 0;
        for (int64_t s2 = n_seg - 1; s2 >= 0; --s2) {
            start[s2] = (uint32_t)pos;
            for (int64_t i = off[s2]; i < off[s2 + 1]; ++i) src[pos++] = data[i];
        }
    } else {
        for (int64_t i = 0; i < n; ++i) src[i] = data[i];
    }
    AMIRA_CUDA(cudaMemcpyAsync(d_a.p, src.data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice, st));
    AMIRA_CUDA(cudaMemcpyAsync(d_start.p, start.data(), sizeof(uint32_t) * (n_seg + 1), cudaMemcpyHostToDevice, st));
    AMIRA_CUDA(cudaMemcpyAsync(d_off.p, off, sizeof(int64_t) * (n_seg + 1), cudaMemcpyHostToDevice, st));
    AMIRA_CUDA(cudaMemcpyAsync(d_cnt.p, cnt, sizeof(cnt), cudaMemcpyHostToDevice, st));
    int rc = run_segsort(h, d_a.as<uint32_t>(), d_b.as<uint32_t>(), d_off.as<int64_t>(),
                         out_of_place ? d_start.as<uint32_t>() : nullptr, out_of_place != 0, d_cnt.as<long long>(), 1, n_seg, n,
                         max_value, d_dups.as<uint32_t>(), d_cnt.as<unsigned long long>() + 1);
    if (rc == AMIRA_OK) {
        AMIRA_CUDA(cudaMemcpyAsync(data, out_of_place ? d_b.p : d_a.p, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, st));
        if (dups) AMIRA_CUDA(cudaMemcpyAsync(dups, d_dups.p, sizeof(uint32_t) * n_seg, cudaMemcpyDeviceToHost, st));
        AMIRA_CUDA(cudaMemcpyAsync(cnt, d_cnt.p, sizeof(cnt), cudaMemcpyDeviceToHost, st));
        AMIRA_CUDA(cudaStreamSynchronize(st));
        if (total_dups) *total_dups = cnt[1];
    }
    for (DevBuf *x : {&d_a, &d_b, &d_off, &d_dups, &d_cnt, &d_start}) x->release();
    return rc;
}

int amira_gmg_comm_init(amira_gmg *h, const void *nccl_unique_id, int rank, int world) {
    AMIRA_TRY(check_handle(h));
    if (world < 1 || world > MAX_WORLD || rank < 0 || rank >= world || !nccl_unique_id) {
        set_error("bad arguments to amira_gmg_comm_init (world must be 1..%d)", MAX_WORLD);
        return AMIRA_E_ARG;
    }
    if (h->comm) {
        comm_destroy(h->comm);
        h->comm = nullptr;
    }
    h->built = false;
    h->rank = 0;
    h->world = 1;
    AMIRA_TRY(comm_create(&h->comm, nccl_unique_id, rank, world));
    if (!h->h_cnt) AMIRA_CUDA(cudaMallocHost((void **)&h->h_cnt, sizeof(long long) * ((size_t)MAX_WORLD * MAX_WORLD + 8)));
    h->rank = rank;
    h->world = world;
    return AMIRA_OK;
}

int amira_gmg_atomic_peak(amira_gmg *h, int64_t table_bytes, int64_t n_ops, double *red_add_per_s, double *cas_per_s,
                          double *load_per_s) {
    AMIRA_TRY(check_handle(h));
    if (table_bytes < 64 || n_ops < 1) return AMIRA_E_ARG;
    DevBuf t;
    AMIRA_TRY(t.reserve((size_t)table_bytes));
    AMIRA_TRY(h->d_maxabs.reserve(16));
    cudaEvent_t a, b;
    AMIRA_CUDA(cudaEventCreate(&a));
    AMIRA_CUDA(cudaEventCreate(&b));
    const int grid = h->n_sm * 8;
    float ms = 0.f;
    for (int which = 0; which < 3; ++which) {
        if (which == 2 && !load_per_s) break;
        float best = 1e30f;
        for (int rep = 0; rep < 4; ++rep) {
            AMIRA_CUDA(cudaMemsetAsync(t.p, 0xFF, (size_t)table_bytes, h->stream));
            AMIRA_CUDA(cudaEventRecord(a, h->stream));
            if (which == 0)
                LAUNCH(h, k_atomic_red, grid, 256, t.as<unsigned int>(), (unsigned long long)(table_bytes / 4),
                       (unsigned long long)n_ops, 0x1234ull + rep);
            else if (which == 1)
                LAUNCH(h, k_atomic_cas, grid, 256, t.as<unsigned long long>(), (unsigned long long)(table_bytes / 8),
                       (unsigned long long)n_ops, 0x1234ull + rep);
            else
                LAUNCH(h, k_random_load, grid, 256, t.as<NodeSlot>(), (unsigned long long)(table_bytes / 32),
                       (unsigned long long)n_ops, 0x1234ull + rep, (unsigned long long *)h->d_maxabs.p);
            AMIRA_CUDA(cudaEventRecord(b, h->stream));
            AMIRA_CUDA(cudaEventSynchronize(b));
            AMIRA_CUDA(cudaEventElapsedTime(&ms, a, b));
            if (rep > 0) best = std::min(best, ms);
        }
        double rate = (double)n_ops / (best * 1e-3);
        if (which == 0 && red_add_per_s) *red_add_per_s = rate;
        if (which == 1 && cas_per_s) *cas_per_s = rate;
        if (which == 2 && load_per_s) *load_per_s = rate;
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    t.release();
    return AMIRA_OK;
}

}  // extern "C"
