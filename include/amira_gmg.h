/* amira_gmg.h -- C ABI of the B200-native GeneMerGraph build (libamira_gmg.so).
 *
 * The upstream project (Danderson123/Amira) is pure Python and has no FFI; the boundary this
 * library slots in behind is the Python class boundary
 *     GeneMerGraph(readDict, kmerSize, gene_positions=None)        amira/construct_graph.py:31-102
 *     GeneMerGraph.filter_graph(minNodeCoverage, minEdgeCoverage)   amira/construct_graph.py:523-540
 *     GeneMerGraph.remove_low_coverage_components(c)                amira/construct_graph.py:950-958
 * reached through build_graph / build_multiprocessed_graph           amira/graph_utils.py:12-14, 105-124.
 * Each entry point below names the upstream code it replaces.  INTEGRATION.md shows the ctypes stub
 * a maintainer adds on the upstream side.
 *
 * Conventions: every function returns an int status (AMIRA_OK == 0); amira_last_error() returns a
 * thread-local message for the last failure.  No exception crosses the ABI.  The caller owns every
 * input and output buffer; the library owns only the opaque handle and its device memory.  One
 * handle per (host thread, device); a handle is not thread-safe, distinct handles may be used
 * concurrently.  All device work of a handle is stream-ordered on the handle's stream.
 *
 * Gene ids: int32, id = strand * rank, strand in {+1,-1}, rank in 1..V = position of the gene name
 * in the vocabulary sorted by int(sha256(pickle.dumps(name))) ascending, so that the signed integer
 * order equals the order of upstream's signed gene hashes (amira/construct_gene.py:91-93) and the
 * canonical orientation of every gene-mer is the one upstream picks (construct_gene_mer.py:15-39).
 */
#ifndef AMIRA_GMG_H
#define AMIRA_GMG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct amira_gmg amira_gmg;

enum {
    AMIRA_OK = 0,
    AMIRA_E_BLANK_GENE = 1,    /* "Gene information is missing"          construct_gene.py:52 */
    AMIRA_E_BAD_STRAND = 2,    /* "Strand information missing for: ..."  construct_gene.py:58 */
    AMIRA_E_EMPTY_NAME = 3,    /* "Gene name information missing ..."    construct_gene.py:62 */
    AMIRA_E_UNKNOWN_GENE = 4,  /* token not in the supplied vocabulary */
    AMIRA_E_PALINDROME = 5,    /* "Gene-mer and reverse complement gene-mer are identical"  construct_gene_mer.py:23 */
    AMIRA_E_EMPTY_GENEMER = 6, /* k == 0 with a non-empty read: "Gene-mer is empty"         construct_gene_mer.py:47 */
    AMIRA_E_MULTI_EDGE = 7,    /* remove_node on a node with two edges to one neighbour: upstream TypeError */
    AMIRA_E_ARG = 8,
    AMIRA_E_STATE = 9,         /* call order violated (e.g. export before build) */
    AMIRA_E_CUDA = 10,
    AMIRA_E_NOMEM = 11,
    AMIRA_E_NCCL = 12
};

/* phases timed with CUDA events on the handle's stream (amira_gmg_phase_ms) */
enum {
    AMIRA_PH_H2D = 0,        /* host -> device copy of the CSR input */
    AMIRA_PH_WINDOWS = 1,    /* per-read window counts + scan */
    AMIRA_PH_INSERT = 2,     /* k_insert_windows: enumerate, canonicalise, hash, node + edge tables */
    AMIRA_PH_ORDER = 3,      /* first-seen ranks of nodes and edges (bitmap + prefix popcount) */
    AMIRA_PH_REMAP = 4,      /* node -> reads offsets, units, partition pass (per-window slot -> node index + records dealt into buckets) */
    AMIRA_PH_INCIDENCE = 5,  /* node -> reads CSR: one CTA per unit sorts its lists in shared memory */
    AMIRA_PH_ADJACENCY = 6,  /* node -> forward/backward edge CSR */
    AMIRA_PH_COMPONENTS = 7, /* connected components */
    AMIRA_PH_FILTER = 8,     /* last filter / component removal */
    AMIRA_PH_EXCHANGE = 9,   /* multi-GPU all-to-all + merge */
    AMIRA_PH_EMIT = 10,      /* edge arrays in first-seen order + union-find (second stream, beside REMAP / INCIDENCE,
                              * as are ADJACENCY and COMPONENTS) */
    AMIRA_PH_INSERT_KERNEL = 11, /* k_insert_windows alone (inside AMIRA_PH_INSERT, which also clears the tables) */
    AMIRA_PH_EMIT_NODES = 12,    /* node arrays in first-seen order */
    AMIRA_PH_EXCHANGE_EDGES = 13, /* multi-GPU: edge half of the exchange (second stream, beside REMAP / INCIDENCE) */
    AMIRA_PH_COUNT = 14
};

const char *amira_last_error(void);
const char *amira_version(void);

/* Gene-call token parsing: "+name" / "-name" -> signed id.  Replaces Gene.__init__ /
 * split_gene_and_strand (construct_gene.py:48-67) and convert_genes (construct_read.py:5-8).
 * Tokens are concatenated UTF-8 with tok_off[n_tok+1] byte offsets; vocabulary names likewise, in
 * SHA-rank order (names already have spaces replaced by '_').  Spaces in a token's name are mapped
 * to '_' before the lookup.  tok_off may be NULL: the tokens are then separated by '\n' in a NUL-terminated
 * blob that must hold exactly n_tok of them.  On error returns the code above and writes the index of the
 * offending token to *bad_token (if non-NULL). */
int amira_vocab_encode(const char *tokens_utf8, const int64_t *tok_off, int64_t n_tok,
                       const char *vocab_utf8, const int64_t *vocab_off, int32_t n_vocab,
                       int32_t *out_signed_ids, int64_t *bad_token);

/* Upstream's dictionary keys in bulk, on the host: int(sha256(pickle.dumps(x)).hexdigest(), 16)
 * (construct_gene.py:5-10) for tuples x of signed 256-bit integers given as 32-byte big-endian
 * magnitudes + sign flags (pickle protocol 4, the default of CPython 3.8-3.13).  tuple_sha: node keys
 * (construct_gene_mer.py:94-97) and anything else tuple-shaped; edge_keys: min over both sign choices
 * (construct_edge.py:104-124) from the node keys and the exported edge arrays.  Outputs are 32-byte
 * big-endian digests. */
int amira_host_tuple_sha(const uint8_t *mags, const int8_t *neg, int64_t n_tuples, int32_t arity, uint8_t *out);
int amira_host_edge_keys(const uint8_t *node_sha, const int32_t *src, const int32_t *tgt, const int8_t *sd,
                         const int8_t *td, int64_t n_edges, uint8_t *out);

int amira_gmg_create(amira_gmg **h, int device, void *cuda_stream /* NULL: library-owned stream */);
void amira_gmg_destroy(amira_gmg *h);

/* optional capacity hints (expected unique nodes / undirected edges); 0 = automatic */
int amira_gmg_reserve(amira_gmg *h, int64_t n_nodes_hint, int64_t n_edges_hint);
int amira_gmg_set_profiling(amira_gmg *h, int enabled);
int amira_gmg_phase_ms(const amira_gmg *h, int phase, float *ms);
int amira_gmg_kernel_launches(const amira_gmg *h, int64_t *n);

/* The build: GeneMerGraph.__init__ (construct_graph.py:45-102) for R reads in CSR form.
 * signed_ids[read_off[R]], read_off[R+1]; pos_start/pos_end (nullable) are per-call read
 * coordinates (gene_positions, construct_read.py:46-52).  input_on_device != 0: the pointers are
 * device pointers valid on the handle's stream (they are borrowed until the next build/destroy).
 * Asynchronous with respect to the host unless a capacity retry is needed; errors detected on the
 * device (AMIRA_E_PALINDROME) are reported by amira_gmg_sync / amira_gmg_sizes / the exports. */
int amira_gmg_build(amira_gmg *h, const int32_t *signed_ids, const int64_t *read_off, int64_t R, int32_t k,
                    const int32_t *pos_start, const int32_t *pos_end, int input_on_device);

/* wait for the handle's stream; returns the deferred status of the last build / filter */
int amira_gmg_sync(amira_gmg *h);

/* sizes of the current (possibly filtered) graph; any pointer may be NULL.  n_incidence / n_fw / n_bw
 * wait for the whole build, the others are known as soon as the tables are (so that a caller can
 * size and start the per-read export while the incidence / adjacency passes still run) */
int amira_gmg_sizes(amira_gmg *h, int64_t *n_nodes, int64_t *n_edges, int64_t *n_windows,
                    int64_t *n_incidence, int64_t *n_fw, int64_t *n_bw, int64_t *n_short);

/* Nodes in upstream `_nodes` insertion order (construct_graph.py:196-212):
 * key[n_nodes*k] canonical signed ids, cov (Node.nodeCoverage), first_dir (direction of the
 * first-seen GeneMer), component (assign_component_ids, :920-927), reads CSR (Node.listOfReads as
 * read indices, ascending), forward / backward edge-index CSR (Node.forwardEdgeHashes /
 * backwardEdgeHashes, construct_node.py:79-101).  Any output pointer may be NULL to skip it. */
int amira_gmg_export_nodes(amira_gmg *h, int32_t *key, uint32_t *cov, int8_t *first_dir, uint32_t *component,
                           int64_t *reads_off, int32_t *reads, int64_t *fw_off, int32_t *fw_edges,
                           int64_t *bw_off, int32_t *bw_edges);

/* Edges in upstream `_edges` insertion order (construct_graph.py:268-277): source / target node
 * index, stored (first-seen) directions, coverage. */
int amira_gmg_export_edges(amira_gmg *h, int32_t *src, int32_t *tgt, int8_t *sd, int8_t *td, uint32_t *cov);

/* Per-read lists (_readNodes / _readNodeDirections / _readNodePositions, construct_graph.py:165-178):
 * win_off[R+1], node_idx[W] (-1 = None after filtering), dir[W] (0 where None), start/end[W]
 * (only if positions were supplied; -1 where None), is_short[R] (_shortReads), to_correct[R]
 * (_readsToCorrect). */
int amira_gmg_export_reads(amira_gmg *h, int64_t *win_off, int32_t *node_idx, int8_t *dir, int32_t *start,
                           int32_t *end, uint8_t *is_short, uint8_t *to_correct);

/* remove_low_coverage_components (construct_graph.py:950-958) and filter_graph (:523-540) */
int amira_gmg_remove_low_coverage_components(amira_gmg *h, uint32_t min_component_cov);
int amira_gmg_filter(amira_gmg *h, uint32_t min_node_cov, uint32_t min_edge_cov);

/* Which nodes / edges the LAST filter or component removal kept: keep flags (1 = kept) indexed by the
 * node / edge order BEFORE that call.  Lets a host mirror delete the same objects instead of
 * re-creating the survivors.  Sizes via amira_gmg_filter_mask_sizes. */
int amira_gmg_filter_mask_sizes(amira_gmg *h, int64_t *n_nodes_before, int64_t *n_edges_before);
int amira_gmg_export_filter_masks(amira_gmg *h, int32_t *node_keep, int32_t *edge_keep);

/* ---- the scans Amira runs right after a build, on the device-resident graph (SURVEY.md 8f) ----
 * read_length_coverages: get_overall_mean_node_coverages (graph_utils.py:299-313): sums[i] = number of
 *   (node, read) incidences whose read has >= min_len[i] gene calls (mean node coverage = sums[i] / n_nodes);
 *   at most 16 thresholds.
 * node_coverage_stats: sum and maximum of Node.nodeCoverage (get_all_node_coverages / get_mean_node_coverage,
 *   construct_graph.py:863-871).
 * junk_read_mask: remove_junk_reads (construct_graph.py:1398-1420): mask[r] = 1 kept, 0 rejected (more than
 *   round(n * (1 - error_rate)) of the read's n windows are None; Python's round-half-even), 2 = short read.
 * nodes_containing: get_nodes_containing (construct_graph.py:223-244) for a set of genes given by rank (1..V).
 * remove_nodes: remove_node (construct_graph.py:463-484) for every node whose flag is set (host flags[n_nodes]):
 *   edges, per-read windows (None) and _readsToCorrect follow as in the filters; AMIRA_E_MULTI_EDGE like upstream.
 * remove_nodes_without_reads_of: remove_non_AMR_associated_nodes (construct_graph.py:2941-2959).
 * linear_steps: the building block of get_linear_path_for_node / remove_short_linear_paths / get_unitigs_in_graph
 *   (construct_graph.py:722-861, 679-720, 2961-2975): Node degree and, per node and side (forward / backward),
 *   upstream's one step along a linear path: next node (-1 none), direction in which it is entered, and whether
 *   the walk continues (target of degree 1 or 2, not the node itself).  It reuses the memory of the filter masks:
 *   after it, amira_gmg_filter_mask_sizes / amira_gmg_export_filter_masks fail with AMIRA_E_STATE until the next
 *   filter or removal.
 * A filter or removal that fails with AMIRA_E_MULTI_EDGE leaves the graph unchanged and usable, without filter masks;
 * after one on a graph without nodes the masks describe zero nodes and zero edges. */
int amira_gmg_read_length_coverages(amira_gmg *h, const int32_t *min_len, int32_t n, int64_t *sums);
int amira_gmg_node_coverage_stats(amira_gmg *h, int64_t *sum_cov, uint32_t *max_cov);
int amira_gmg_junk_read_mask(amira_gmg *h, double error_rate, uint8_t *mask);
int amira_gmg_nodes_containing(amira_gmg *h, const int32_t *ranks, int32_t n, uint8_t *flags);
int amira_gmg_remove_nodes(amira_gmg *h, const uint8_t *remove_flags);
int amira_gmg_remove_nodes_without_reads_of(amira_gmg *h, const int32_t *ranks, int32_t n);
int amira_gmg_linear_steps(amira_gmg *h, uint32_t *degree, int32_t *fw_next, int8_t *fw_dir, uint8_t *fw_ext,
                           int32_t *bw_next, int8_t *bw_dir, uint8_t *bw_ext);

/* Multi-GPU (one process per GPU; no upstream counterpart -- upstream's joblib fan-out,
 * graph_utils.py:105-124, is disabled at every call site).  The globally ordered read set is
 * sharded contiguously over ranks in rank order; canonical gene-mers and edges are owned by hash
 * range and the partial tables are routed with NCCL all-to-alls.  nccl_unique_id is the 128-byte
 * ncclUniqueId created by rank 0 (amira_gmg_nccl_unique_id) and distributed by the caller.  After
 * comm_init every amira_gmg_build is COLLECTIVE: each rank passes its own shard, and ends with the
 * identical global node / edge tables (exports as on one GPU); the per-read exports and the
 * node -> read incidence cover the rank's own reads, read indices are global.  Filters are
 * collective-free (every rank applies them to the replicated tables). */
int amira_gmg_nccl_unique_id(void *out_128_bytes);
int amira_gmg_comm_init(amira_gmg *h, const void *nccl_unique_id, int rank, int world);

/* Test hook: forbid table layouts the library would otherwise choose from the input, so that the
 * rarely taken ones are exercised at small sizes.  mask bits: 1 = no 16-byte node slots, 2 = no
 * 16-byte edge slots, 4 = no packed keys (gene-mers compared through the ids array), 8 = the 16384-bucket
 * shape of the partition pass, 16 = units of the node -> reads transpose share buckets. */
int amira_gmg_debug_layout(amira_gmg *h, int mask);

/* Test hook: the segmented sort behind the node -> reads and node -> edges lists, on host arrays:
 * data[off[s] .. off[s+1]) is sorted ascending for every s < n_seg (values < max_value); dups[s] (nullable)
 * receives the number of equal neighbours in segment s, *total_dups their sum.  out_of_place != 0 runs the
 * variant that reads the segments from a differently ordered source buffer (odd number of radix passes). */
int amira_gmg_debug_segsort(amira_gmg *h, uint32_t *data, const int64_t *off, int64_t n_seg, uint32_t *dups,
                            int64_t *total_dups, int out_of_place, int64_t max_value);

/* Micro-benchmark for the atomic roofline (SURVEY.md 8d): random-address 32-bit RED.ADD, 64-bit CAS
 * and (if load_per_s is non-NULL) 32-byte sector loads into a table of table_bytes; returns
 * operations per second of each. */
int amira_gmg_atomic_peak(amira_gmg *h, int64_t table_bytes, int64_t n_ops, double *red_add_per_s,
                          double *cas_per_s, double *load_per_s);

#ifdef __cplusplus
}
#endif
#endif /* AMIRA_GMG_H */
