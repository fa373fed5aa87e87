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
 * device pointers valid on the handle's stream (they are borrowed until the next build/destroy).  A device build
 * remembers read_off[R] for the next build only: that build reuses it when it gets the same read_off and R, which
 * the borrow makes the same array; any other build copies read_off[R] back unless amira_gmg_input_calls gave it.
 * Asynchronous with respect to the host unless a capacity retry is needed; errors detected on the
 * device (AMIRA_E_PALINDROME) are reported by amira_gmg_sync / amira_gmg_sizes / the exports. */
int amira_gmg_build(amira_gmg *h, const int32_t *signed_ids, const int64_t *read_off, int64_t R, int32_t k,
                    const int32_t *pos_start, const int32_t *pos_end, int input_on_device);

/* The call count of the NEXT amira_gmg_build only, for a device CSR (input_on_device) whose read_off[R] the caller
 * already knows, such as the outputs of amira_gmg_correct_bubble_reads (n_calls).  That build uses n_calls when it
 * gets the same read_off and R, instead of copying read_off[R] back to the host.  The per-read pass still checks the
 * count on the device.  Every build forgets the hint, used or not.
 * AMIRA_E_ARG for a NULL read_off, R <= 0 or a negative n_calls. */
int amira_gmg_input_calls(amira_gmg *h, const int64_t *read_off, int64_t R, int64_t n_calls);

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

/* Linear walks (get_forward_path_from_node / get_backward_path_from_node, construct_graph.py:722-848) from n start
 * states (2*node + side, side 0 = forward list, 1 = backward list), without the start node, in walk order, plus the
 * branching node when want_branched.  walk_nodes == NULL: only walk_off[n+1] is written (sizes); then call again with
 * walk_nodes[walk_off[n]].  Leaves the filter masks alone.  AMIRA_E_STATE for a walk that never ends.
 * The walk from s0 (node n0) follows succ(s) = 2*next[s] + (dir[s] == 1 ? 0 : 1) while ext[s] is set (linear_steps),
 * and stops before a state of n0; the branching node is next[s] of the state it stopped on, when there is one.
 * Not available on a sharded handle (AMIRA_E_STATE). */
int amira_gmg_linear_walks(amira_gmg *h, const int32_t *states, int64_t n, int want_branched, int64_t *walk_off,
                           int32_t *walk_nodes);

/* The compacted graph: every maximal non-branching path as one unitig (no upstream counterpart).  With states
 * s = 2*node + side as above, succ(2u + a) = 2v + (td == 1 ? 0 : 1) when list a of u holds exactly one edge
 * (u -> v, td), v != u, and v's entering list (backward if td == +1, forward if td == -1) holds exactly one edge.
 * The states form disjoint paths and cycles; a chain with its mirror (every state ^ 1) is one unitig, and every node
 * lies in exactly one.  A unitig is listed in the orientation whose chain holds 2m, m its smallest node: a linear one
 * from its head (the state without predecessor) to its tail, a circular one from m.  Unitig ids follow m ascending.
 *   per node [N]: node_unitig, node_pos (position in the listed order), node_orient (+1: left through its forward
 *     list in that order, -1: through its backward list);
 *   per unitig [U]: unitig_off[U+1] into unitig_nodes[N] (node indices in listed order), circular, cov_sum /
 *     cov_min / cov_max of the node coverages;
 *   per directed edge [E]: edge_internal = 1 when the edge joins consecutive nodes of one unitig (in either
 *     direction); the others are the junctions.  There are 2 * (N - linear unitigs) internal edges.
 * Every pointer may be NULL.  Call with n_unitigs only to size the per-unitig arrays, then again for the arrays: the
 * result is kept on the device until the next build, filter or node removal.  Leaves the filter masks alone.
 * Not available on a sharded handle (AMIRA_E_STATE); AMIRA_E_ARG for 2N >= 2^31. */
int amira_gmg_unitigs(amira_gmg *h, int64_t *n_unitigs, int32_t *node_unitig, int32_t *node_pos, int8_t *node_orient,
                      int64_t *unitig_off, int32_t *unitig_nodes, uint8_t *circular, int64_t *cov_sum, uint32_t *cov_min,
                      uint32_t *cov_max, uint8_t *edge_internal);

/* The edges and the reads of the compacted graph (no upstream counterpart), over the unitigs of amira_gmg_unitigs
 * (node_unitig, node_pos, node_orient and succ as above; reused while cached, not ranked again).  A directed edge
 * j = (u -> v, sd, td) leaves u through the state 2u + (sd < 0); a read window on node n with direction d leaves n
 * through 2n + (d < 0) (the build makes the edge between two windows with the first one's direction as sd).
 * An orientation of +1 means in the unitig's listed order.
 *
 * Links: one per junction edge (edge_internal == 0), in edge order, E - sum(edge_internal) of them:
 *   edge = j, from_unitig = node_unitig[u], from_orient = sd * node_orient[u], to_unitig = node_unitig[v],
 *   to_orient = td * node_orient[v], cov = the edge's coverage.
 *   With from_orient = +1, u is the last node of its unitig, with -1 the first; likewise v at the entering end
 *   (+1: first, -1: last).  No link touches a circular unitig.  Every link (a, oa) -> (b, ob) has its twin
 *   (b, -ob) -> (a, -oa) from the reverse edge (a self edge may be its own twin).
 *
 * Read paths: per read, in read order, its steps.  A step is a maximal run of consecutive windows i..j of one read,
 * all live (not None), each continuing the one before: succ(state(i')) == state(i' + 1).  Equivalently: one unitig,
 * one orientation, and the position moves by one in the direction of travel (modulo the length of a circular
 * unitig, which a read may go round more than once: a step may be longer than its unitig).  A None window belongs
 * to no step and ends the current one.  Per step:
 *   unitig, orient = d * node_orient[n] of its first window (constant along the step), pos = node_pos of the first
 *   window's node, win = the first window's index within the read (as in _readNodes[read]), length = its windows.
 *   path_off[R+1] delimits each read's steps (path_off[R] = the number of steps); short reads and reads whose
 *   windows are all None have empty paths.
 *
 * Both calls: every pointer may be NULL.  Call with n_links only, or path_off only, to size the outputs, then again
 * for the arrays: the results are kept on the device until the next build, filter or node removal.  Leave the
 * filter masks alone.  Not available on a sharded handle (AMIRA_E_STATE); AMIRA_E_ARG for 2N >= 2^31. */
int amira_gmg_unitig_links(amira_gmg *h, int64_t *n_links, int32_t *edge, int32_t *from_unitig, int8_t *from_orient,
                           int32_t *to_unitig, int8_t *to_orient, uint32_t *cov);
int amira_gmg_read_unitig_paths(amira_gmg *h, int64_t *path_off, int32_t *unitig, int8_t *orient, int32_t *pos,
                                int32_t *win, int32_t *length);

/* The simple bubbles of the compacted graph (no upstream counterpart): two or more unitigs that leave one junction
 * and rejoin the graph at another, as one wrong gene call in one read makes (a run of about k wrong gene-mers beside
 * the true path).  Over the unitigs of amira_gmg_unitigs and the read paths of amira_gmg_read_unitig_paths (reused
 * while cached, not ranked again).
 *
 * A state is s = 2 * node + side; list(s) is that node's forward (side 0) or backward (side 1) list.  A directed
 * edge e = (u -> v, sd, td) lies in list(2u + (sd < 0)); it continues through cont(e) = 2v + (td < 0), the state a
 * walk leaves v through, and v's entering list for e is list(cont(e) ^ 1).
 *
 * Branch: an edge e in list(sigma), x = sigma >> 1, with target h, enters the branch b = the unitig of h when
 *   1. list(cont(e) ^ 1) holds exactly one edge;
 *   2. b is not circular;
 *   3. the walk through b from h in the direction of cont(e) reaches b's other end node t, t is left through s_t,
 *      and list(s_t) holds exactly one edge e', with target y;
 *   4. neither x nor y is a node of b.
 * (With 1. and x not in b, h has no predecessor in b: it is b's end on the entering side, and the branch is all of b.)
 * The branch runs from sigma to tau = cont(e').  Its orientation is +1 when h is the first node of b in listed
 * order (always for a one-node b), -1 otherwise.
 * Bubble: the branches of list(sigma) grouped by tau; a group of two or more with sigma < (tau ^ 1) is one bubble.
 * With sigma > (tau ^ 1) the same bubble is reported from tau ^ 1 (its mirror); with sigma == (tau ^ 1) the branches
 * only turn back into the end they left, and there is no bubble.  So every bubble is reported once, and a unitig is
 * a branch of at most one bubble.
 *
 * Outputs, in an order that does not depend on thread timing: bubbles by sigma ascending, then by the list(sigma)
 * position of their first branch; branches in list(sigma) order (upstream's forward / backward list order).
 *   per bubble: source = sigma, sink = tau (states); branch_off[B+1] delimits its branches;
 *   per branch: branch_unitig, branch_orient, branch_reads = the read steps (amira_gmg_read_unitig_paths) on the
 *   unitig whose length equals its node count: the reads that run the whole branch, in either direction.
 * Lengths and coverages are those of amira_gmg_unitigs (unitig_off, cov_sum, ...), not copied here.
 *
 * Out of scope: bubbles whose branches are not single unitigs (nested or overlapping errors, superbubbles), and
 * branches without a node (an edge joining the two junction nodes directly, as a deletion makes at k = 1).
 *
 * Every pointer may be NULL.  Call with n_bubbles / n_branches only to size the outputs, then again for the arrays:
 * the result is kept on the device until the next build, filter or node removal.  Leaves the filter masks alone.
 * Not available on a sharded handle (AMIRA_E_STATE); AMIRA_E_ARG for 2N >= 2^31.  Grouping a list of d edges takes
 * O(d^2 / 32) warp steps. */
int amira_gmg_bubbles(amira_gmg *h, int64_t *n_bubbles, int64_t *n_branches, int32_t *source, int32_t *sink,
                      int64_t *branch_off, int32_t *branch_unitig, int8_t *branch_orient, uint32_t *branch_reads);

/* The reads through the simple bubbles of amira_gmg_bubbles rewritten along a kept branch (no upstream counterpart,
 * like the popping policy): the correction step of a "pop, correct, rebuild" cleaning loop, computed from the build's
 * input CSR (kept or borrowed by amira_gmg_build), the cached read paths and bubbles, and the node keys.
 *
 * replace_with[n_branches] (host): per branch g of amira_gmg_bubbles, -1 leaves g's reads alone; otherwise it is
 * another branch of the same bubble, whose genes replace g's calls.  NULL: the replace_with the last
 * amira_gmg_bubble_policy left on the device, used without a host check (it is valid by construction); AMIRA_E_STATE
 * when there are branches and no policy was computed on the current bubbles (a build, filter or node removal came
 * since, or a call with a host replace_with overwrote it).
 * Edit: a read step (amira_gmg_read_unitig_paths) on branch g = unitig b of m nodes in bubble (sigma, tau), with
 * replace_with[g] >= 0, length m, the windows win - 1 and win + m present in its read and live, and their states
 * (2 * node + (dir < 0)) either (sigma, tau) -- the read runs sigma -> b -> tau -- or (tau ^ 1, sigma ^ 1) -- the
 * mirror.  (The state check matters: a filter with min_edge_cov > 1 can delete the edge between two live windows.)
 * Rewrite: window i of a read starts at its call i.  An edit replaces the m calls [win, win + m) by m' calls, m' the
 * kept branch's node count; call j is the first gene of the j-th kept node in the direction of travel: the kept
 * branch is walked in listed order when (+1 for sigma -> tau, -1 for the mirror) * its branch_orient is +1, a node
 * n's direction along the walk is node_orient[n] in listed order and -node_orient[n] against it, and its first gene
 * is key[n * k] in direction +1, -key[n * k + k - 1] in direction -1.  The read then spells source, kept branch,
 * sink.  Edits never overlap, and two edits of one read have an untouched call between them: every node of a branch
 * has one-edge lists on both sides, a junction node a list of two edges or more.
 * Positions (without positions pos_start / pos_end are ignored): untouched calls keep theirs; new call j < m takes
 * those of replaced call j, new call j >= m those of the last replaced call.
 * Everything else is unchanged: steps that do not qualify (a full-length step without both flanks, as a read that
 * starts or ends on the branch, counts in branch_reads but is not rewritten), short reads, reads without an edit.
 *
 * Outputs: n_calls = the new call count; read_off[R + 1], ids / pos_start / pos_end [n_calls] the corrected CSR in
 * read order (read_off[r] = the output index of the input's call read_off_in[r]); changed[R] = 1 for a read with an
 * edit; branch_rewritten[n_branches] = the edits per branch.  Call with n_calls only to size the outputs, then again
 * for the arrays; every output may be NULL.  out_on_device != 0: the array outputs are device pointers on the handle's
 * device; either way the call returns with the work complete, and the library keeps no pointer.  A build from device
 * outputs can be given n_calls with amira_gmg_input_calls, so that it copies nothing back to size itself.  Leaves the
 * graph,
 * the cached unitigs / paths / bubbles and the filter masks as they were.  AMIRA_E_ARG when replace_with points out
 * of range, into another bubble or at the branch itself; AMIRA_E_STATE on a sharded handle.  Out of scope: reads that
 * end inside a branch, nested bubbles and superbubbles. */
int amira_gmg_correct_bubble_reads(amira_gmg *h, const int32_t *replace_with, int64_t *n_calls, int64_t *read_off,
                                   int32_t *ids, int32_t *pos_start, int32_t *pos_end, uint8_t *changed,
                                   uint32_t *branch_rewritten, int out_on_device);

/* The popping policy of the simple bubbles (no upstream counterpart; GeneMerGraph.pop_compacted_bubbles and
 * correct_compacted_bubbles use it), over the cached unitigs and bubbles, computed if not cached.  Per bubble the kept
 * branch has the largest mean node coverage cov_sum / length of its unitig (amira_gmg_unitigs), compared exactly by
 * cross-multiplying in 128 bits; ties go to the most branch_reads, then to the lowest branch index.  Every other
 * branch is replaced by the kept one (replace_with[g] = the kept branch), unless one of its nodes holds a gene of
 * spare_ranks[n_ranks] (vocabulary ranks as amira_gmg_nodes_containing takes them): then, as for the kept branch,
 * replace_with[g] = -1.
 *
 * Outputs: n_replaced = the branches replaced; replace_with[n_branches] (host, may be NULL).  The result stays on the
 * device, tagged with the bubble cache it belongs to, for amira_gmg_correct_bubble_reads with replace_with == NULL.
 * One warp per bubble, whatever its branch count.  AMIRA_E_ARG for bad ranks; AMIRA_E_STATE on a sharded handle.
 * Leaves the graph, the caches and the filter masks as they were. */
int amira_gmg_bubble_policy(amira_gmg *h, const int32_t *spare_ranks, int32_t n_ranks, int64_t *n_replaced,
                            int32_t *replace_with);

/* The dead-end tips of the compacted graph (no upstream counterpart): the short chain of wrong gene-mers an error in
 * the first or last k calls of a read makes, which leaves the true path at a junction and stops at the read's end.
 * Over the unitigs of amira_gmg_unitigs and the read paths of amira_gmg_read_unitig_paths (reused while cached, not
 * ranked again).  States, list(s) and cont(e) as for amira_gmg_bubbles; a read window on node n with direction d is in
 * state 2n + (d < 0).
 *
 * Tip: a non-circular unitig b, h0 its first node and h1 its last in listed order (one node for a one-node unitig),
 * with its two outward end states out1 = 2 * h1 + (node_orient[h1] < 0) (leaving h1 in listed order) and
 * out0 = (2 * h0 + (node_orient[h0] < 0)) ^ 1 (leaving h0 against it), such that
 *   1. exactly one of list(out0) and list(out1) is empty (the dead end), and
 *   2. the other one, list(s_t), holds exactly one edge e', whose target v is not a node of b.
 * By maximality list(attach) then holds two edges or more.  A unitig with both ends dead (a linear component) or both
 * ends attached (a possible bubble branch) is no tip.
 * Per tip, in ascending unitig order: tip_unitig = b; tip_orient = +1 when a walk from v into b follows b's listed
 * order (the dead end is out1), -1 otherwise (for a one-node tip too: it depends on which state is dead);
 * tip_attach = cont(e') ^ 1, the state a walk leaves v through into the tip; tip_reads = the read steps on b.
 *
 * Every pointer may be NULL.  Call with n_tips only to size the outputs, then again for the arrays: the result is
 * kept on the device until the next build, filter or node removal.  Leaves the filter masks alone.  Not available on a
 * sharded handle (AMIRA_E_STATE); AMIRA_E_ARG for 2N >= 2^31. */
int amira_gmg_tips(amira_gmg *h, int64_t *n_tips, int32_t *tip_unitig, int8_t *tip_orient, int32_t *tip_attach,
                   uint32_t *tip_reads);

/* The clipping policy of the tips (no upstream counterpart), over the cached tips and unitigs, computed if not cached.
 * Tip q on unitig b, attached at alpha = tip_attach[q], is clipped (clip[q] = 1, else 0) when
 *   1. b has fewer than min_length nodes;
 *   2. no node of b holds a gene of spare_ranks[n_ranks] (vocabulary ranks as amira_gmg_nodes_containing takes them);
 *   3. some edge of list(alpha) whose target w is not on b leads into a unitig c with a strictly larger mean node
 *      coverage: cov_sum[c] * len(b) > cov_sum[b] * len(c), compared exactly in 128 bits.  Equal means: not clipped.
 * Condition 3 matters: the true path's own last unitig is often a dead end on the same junction, and so a tip too; it
 * stays because its coverage is higher.  An error in the last (or first) k calls of a read makes a tip of at most k
 * nodes, so min_length = k + 1 covers single end errors.
 *
 * Outputs: n_clipped = the tips clipped; clip[n_tips] (host, may be NULL).  The flags stay on the device, tagged with
 * the tip cache they belong to, for amira_gmg_clip_tip_reads with clip == NULL.  One warp per tip scans list(alpha):
 * d tips on one list of d edges cost O(d^2) in all.  AMIRA_E_ARG for bad ranks; AMIRA_E_STATE on a sharded handle.
 * Leaves the graph, the caches and the filter masks as they were. */
int amira_gmg_tip_policy(amira_gmg *h, int32_t min_length, const int32_t *spare_ranks, int32_t n_ranks,
                         int64_t *n_clipped, uint8_t *clip);

/* The reads that run into clipped tips, clipped (no upstream counterpart): the tip counterpart of
 * amira_gmg_correct_bubble_reads, from the build's input CSR and the cached read paths and tips.
 *
 * clip[n_tips] (host): 1 clips tip q, 0 leaves it; any other value is AMIRA_E_ARG.  NULL: the flags the last
 * amira_gmg_tip_policy left on the device; AMIRA_E_STATE when there are tips and no policy was computed on the current
 * tips (a build, filter or node removal came since, or a call with host flags overwrote them).
 * Clip: a read step (win = i, length = l) of read r with nw windows on the unitig of a clipped tip attached at alpha:
 *   end clip:   i >= 1, i + l == nw, window i - 1 live with state alpha: the read's last l calls are dropped;
 *   start clip: i == 0, l < nw, window l live with state alpha ^ 1: the read's first l calls are dropped.
 * Window i covers calls [i, i + k), so the dropped calls are exactly those only tip windows hold; positions go with
 * their calls.  A read may have a start clip and an end clip; they never overlap, and a clipped read keeps at least
 * one window (k calls or more).  Left alone: a read lying wholly on a tip, a step that does not reach the read's end
 * (None windows follow it), a flank window whose state does not match (a filter with min_edge_cov > 1 can do that),
 * short reads, every other call and read.
 *
 * Outputs as amira_gmg_correct_bubble_reads: n_calls; read_off[R + 1], ids / pos_start / pos_end [n_calls], the
 * clipped CSR in read order; changed[R] = 1 for a clipped read; tip_clipped[n_tips] = the steps clipped per tip.  Call
 * with n_calls only to size the outputs, then again for the arrays; every output may be NULL.  out_on_device != 0: the
 * array outputs are device pointers on the handle's device; a build from them can be given n_calls with
 * amira_gmg_input_calls.  Leaves the graph, the caches and the filter masks as they were; AMIRA_E_STATE on a sharded
 * handle. */
int amira_gmg_clip_tip_reads(amira_gmg *h, const uint8_t *clip, int64_t *n_calls, int64_t *read_off, int32_t *ids,
                             int32_t *pos_start, int32_t *pos_end, uint8_t *changed, uint32_t *tip_clipped,
                             int out_on_device);

/* The reads cleaned of bubbles and tips in one pass (no upstream counterpart; one iteration of the read corrections of
 * upstream's iterative_bubble_popping, graph_utils.py:127-181): the edits of amira_gmg_correct_bubble_reads and the
 * clips of amira_gmg_clip_tip_reads, applied to the same graph and written as one CSR.
 *
 * The two never touch the same call.  An edit rewrites calls [win, win + m) strictly inside a read, on the windows of
 * a branch, and its flanking windows win - 1 and win + m are live windows on the bubble's junction nodes.  A clip
 * drops the calls only tip windows hold, at a read's first or last step.  A branch unitig has one-edge lists at both
 * ends; a tip unitig has a dead end, and its attach node has a list of two edges or more, so it lies on no branch.  No
 * unitig is both a branch and a tip, so no window is, and the dropped calls of a clip (held by tip windows alone) are
 * no call of an edit, whose windows lie on a branch or are its flanks on junction nodes.
 *
 * replace_with[n_branches] and clip[n_tips] (host) as the two calls take them, checked the same way (AMIRA_E_ARG),
 * and overwriting the held policy the same way; NULL takes the held policy, AMIRA_E_STATE when there are branches
 * (tips) and no bubble (tip) policy was computed on the current bubbles (tips).  Both are checked before any device
 * work.  Outputs as the two calls: n_calls; read_off[R + 1], ids / pos_start / pos_end [n_calls]; changed[R] = 1 for a
 * read edited or clipped; branch_rewritten[n_branches] and tip_clipped[n_tips].  Every output may be NULL; out_on_device
 * and amira_gmg_input_calls as for the two calls.  Leaves the graph, the caches, both held policies and the filter
 * masks as they were; AMIRA_E_STATE on a sharded handle. */
int amira_gmg_clean_reads(amira_gmg *h, const int32_t *replace_with, const uint8_t *clip, int64_t *n_calls,
                          int64_t *read_off, int32_t *ids, int32_t *pos_start, int32_t *pos_end, uint8_t *changed,
                          uint32_t *branch_rewritten, uint32_t *tip_clipped, int out_on_device);

/* The reads grouped by their path through the genes of interest (no upstream counterpart as one call; the nearest
 * relative is assign_reads_to_genes with get_AMR_anchors and get_full_paths, construct_graph.py:2629-2691, 2725-2782,
 * 2880-2939).  Over the per-read windows of the graph as it stands (built, filtered, nodes removed: amira_gmg_export_reads),
 * not the compacted graph.
 *
 * Marked node: one that holds a gene of ranks[n_ranks] (vocabulary ranks, checked as amira_gmg_nodes_containing checks
 * them).  A window of read r (index i in 0..nw-1) is live when its node is >= 0; its state is 2 * node + (dir < 0).
 * Occurrence: a maximal run of windows i..j of one read, all live and on marked nodes; occurrences are numbered in
 * global window order (read, then window).  It has a left flank when i >= 1 and window i - 1 is live (unmarked, by
 * maximality), a right flank when j + 1 < nw and window j + 1 is live; with both it is complete, else partial.
 * Span S: the states of windows i - 1 (with a left flank) .. j + 1 (with a right flank), in read order.  R(S) is S
 * reversed with every state ^ 1; the canonical sequence is the lexicographically smaller of S and R(S) (int32
 * sequences); occ_orient = +1 when S <= R(S), -1 otherwise.
 * Clusters: the complete occurrences grouped by canonical sequence, numbered by their first occurrence; key(c) is that
 * sequence.  A partial occurrence whose S or R(S) is a contiguous subsequence of the key of exactly one cluster c gets
 * occ_cluster = c and occ_orient = +1 when S itself occurs in key(c), else -1; of no cluster -1, of two or more -2
 * (ambiguous), both keeping the orientation of their own canonical sequence.  A complete occurrence's occ_cluster is
 * its cluster.  Members of c: its complete occurrences and the partial ones assigned to it, ascending.
 *
 * Outputs, in an order that does not depend on thread timing or on the key hash:
 *   per occurrence [n_occurrences]: occ_read, occ_win (its first window's index within the read, as in _readNodes),
 *     occ_length (windows), occ_flanks (1 left, 2 right), occ_orient, occ_cluster;
 *   per cluster [n_clusters]: key_off[C + 1] into key_state[n_key_states], n_complete (its complete occurrences),
 *     member_off[C + 1] into members[n_members] (occurrence indices).
 * Every pointer may be NULL.  Call with the counts only to size the outputs, then again for the arrays: the result is
 * kept on the device, with the ranks it was computed for, until the next build, filter or node removal; a call with the
 * same ranks launches nothing.  Leaves the graph, the filter masks, the other caches and both held policies as they were.
 * Not available on a sharded handle (AMIRA_E_STATE); AMIRA_E_ARG for bad ranks and for more than 2^31 - 1 occurrences.
 * Matching a partial occurrence walks the key entries of the node of its first state: O(partials x entries of that
 * node x span length).  Out of scope: clusters that differ by a call error (clean the reads first, or threshold on the
 * member counts), context beyond one flank window, one cluster set per gene (call once per gene). */
int amira_gmg_gene_paths(amira_gmg *h, const int32_t *ranks, int32_t n_ranks, int64_t *n_occurrences, int64_t *n_clusters,
                         int64_t *n_key_states, int64_t *n_members, int32_t *occ_read, int32_t *occ_win, int32_t *occ_length,
                         uint8_t *occ_flanks, int8_t *occ_orient, int32_t *occ_cluster, int64_t *key_off, int32_t *key_state,
                         uint32_t *n_complete, int64_t *member_off, int32_t *members);

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
 * shape of the partition pass, 16 = units of the node -> reads transpose share buckets, 32 = amira_gmg_gene_paths
 * cuts its key hash to 3 bits (every probe of its table then compares sequences; the outputs do not change). */
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
