/* CPU oracle (plain C) for Amira's gene-space de Bruijn graph build -- TEST INFRASTRUCTURE ONLY.
 *
 * The checker, never the product: only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load this library.  Nothing under amira_b200/ links it.
 *
 * Single-threaded scalar restatement on integer gene ids (id = strand * SHA-rank, so that signed
 * integer order equals the reference's signed SHA-256 order, construct_gene.py:91-93):
 *   - window enumeration                       amira/construct_read.py:37-59
 *   - reverse complement, canonical, direction amira/construct_gene_mer.py:4-39, 60-70
 *   - the build loop                           amira/construct_graph.py:45-100
 *   - add_node / add_node_to_read / add_edge   amira/construct_graph.py:165-178, 196-212, 246-324
 *   - edge identity                            amira/construct_edge.py:104-124
 *   - node read list (unique, first touch)     amira/construct_node.py:64-67
 *   - component numbering                      amira/construct_graph.py:911-927
 *   - filter_graph / remove_low_coverage_components   amira/construct_graph.py:409-540, 929-958
 *   - remove_node for a set of nodes           amira/construct_graph.py:463-484
 *
 * It follows the reference's *event order* literally (forward edge then reverse edge per adjacent
 * pair, each one insert-or-get followed by a coverage increment) rather than any derived shortcut,
 * so that it is an independent check of the shortcuts the CUDA path takes.
 *
 * Parity status: PINNED -- tests/test_oracle_golden.py checks it against the golden vectors that
 * oracle/make_golden.py produced by running the unmodified upstream GeneMerGraph.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORACLE_OK 0
#define ORACLE_E_PALINDROME 1
#define ORACLE_E_NOMEM 2
#define ORACLE_E_MULTIEDGE 3
#define ORACLE_E_BADARG 4

typedef struct {
    int32_t k;
    int64_t R, W;
    /* nodes (insertion order) */
    int64_t n_nodes, cap_nodes;
    int32_t *node_key;       /* n_nodes * k */
    uint32_t *node_cov;
    int8_t *node_dir;
    uint32_t *node_comp;
    int32_t *node_last_read;
    /* node hash map: slot -> node idx or -1 */
    int64_t map_cap;
    int32_t *map;
    /* incidence pairs in event order */
    int64_t n_inc, cap_inc;
    int32_t *inc_node, *inc_read;
    /* edges (insertion order) */
    int64_t n_edges, cap_edges;
    int32_t *edge_src, *edge_tgt;
    int8_t *edge_sd, *edge_td;
    uint32_t *edge_cov;
    int64_t emap_cap;
    int32_t *emap;
    /* per window */
    int64_t *win_off;        /* R+1 */
    int32_t *win_node;
    int8_t *win_dir;
    int32_t *win_start, *win_end;
    uint8_t *is_short, *to_correct;
} oracle_graph;

static uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

static uint64_t hash_key(const int32_t *key, int k) {
    uint64_t h = 0x9e3779b97f4a7c15ULL;
    for (int j = 0; j < k; ++j) h = mix64(h ^ (uint64_t)(uint32_t)key[j]);
    return h;
}

static int grow_nodes(oracle_graph *g) {
    int64_t cap = g->cap_nodes ? g->cap_nodes * 2 : 1024;
    int kk = g->k > 0 ? g->k : 1;
    g->node_key = realloc(g->node_key, sizeof(int32_t) * cap * kk);
    g->node_cov = realloc(g->node_cov, sizeof(uint32_t) * cap);
    g->node_dir = realloc(g->node_dir, cap);
    g->node_comp = realloc(g->node_comp, sizeof(uint32_t) * cap);
    g->node_last_read = realloc(g->node_last_read, sizeof(int32_t) * cap);
    if (!g->node_key || !g->node_cov || !g->node_dir || !g->node_comp || !g->node_last_read) return 0;
    g->cap_nodes = cap;
    return 1;
}

static int rehash_nodes(oracle_graph *g) {
    int64_t cap = g->map_cap ? g->map_cap * 2 : 4096;
    int32_t *m = malloc(sizeof(int32_t) * cap);
    if (!m) return 0;
    memset(m, 0xff, sizeof(int32_t) * cap);
    for (int64_t i = 0; i < g->n_nodes; ++i) {
        uint64_t s = hash_key(g->node_key + i * g->k, g->k) & (uint64_t)(cap - 1);
        while (m[s] >= 0) s = (s + 1) & (uint64_t)(cap - 1);
        m[s] = (int32_t)i;
    }
    free(g->map);
    g->map = m;
    g->map_cap = cap;
    return 1;
}

/* insert-or-get a node by canonical key; returns idx or -1 on OOM */
static int32_t node_get(oracle_graph *g, const int32_t *key, int8_t dir) {
    if ((g->n_nodes + 1) * 2 > g->map_cap && !rehash_nodes(g)) return -1;
    uint64_t s = hash_key(key, g->k) & (uint64_t)(g->map_cap - 1);
    while (g->map[s] >= 0) {
        if (memcmp(g->node_key + (int64_t)g->map[s] * g->k, key, sizeof(int32_t) * g->k) == 0) return g->map[s];
        s = (s + 1) & (uint64_t)(g->map_cap - 1);
    }
    if (g->n_nodes == g->cap_nodes && !grow_nodes(g)) return -1;
    int32_t i = (int32_t)g->n_nodes++;
    memcpy(g->node_key + (int64_t)i * g->k, key, sizeof(int32_t) * g->k);
    g->node_cov[i] = 0;
    g->node_dir[i] = dir;          /* Node.geneMer = first-seen GeneMer (construct_node.py:5-7) */
    g->node_comp[i] = 0;
    g->node_last_read[i] = -1;
    g->map[s] = i;
    return i;
}

static int node_touch(oracle_graph *g, int32_t n, int32_t read) {
    /* Node.add_read: unique, first-touch order; reads arrive in ascending order */
    if (g->node_last_read[n] == read) return 1;
    g->node_last_read[n] = read;
    if (g->n_inc == g->cap_inc) {
        int64_t cap = g->cap_inc ? g->cap_inc * 2 : 4096;
        g->inc_node = realloc(g->inc_node, sizeof(int32_t) * cap);
        g->inc_read = realloc(g->inc_read, sizeof(int32_t) * cap);
        if (!g->inc_node || !g->inc_read) return 0;
        g->cap_inc = cap;
    }
    g->inc_node[g->n_inc] = n;
    g->inc_read[g->n_inc] = read;
    g->n_inc++;
    return 1;
}

static uint64_t edge_hash(int32_t s, int32_t t, int rel) {
    return mix64(((uint64_t)(uint32_t)s << 32 | (uint32_t)t) * 2 + (rel > 0));
}

static int rehash_edges(oracle_graph *g) {
    int64_t cap = g->emap_cap ? g->emap_cap * 2 : 4096;
    int32_t *m = malloc(sizeof(int32_t) * cap);
    if (!m) return 0;
    memset(m, 0xff, sizeof(int32_t) * cap);
    for (int64_t i = 0; i < g->n_edges; ++i) {
        uint64_t s = edge_hash(g->edge_src[i], g->edge_tgt[i], g->edge_sd[i] * g->edge_td[i]) & (uint64_t)(cap - 1);
        while (m[s] >= 0) s = (s + 1) & (uint64_t)(cap - 1);
        m[s] = (int32_t)i;
    }
    free(g->emap);
    g->emap = m;
    g->emap_cap = cap;
    return 1;
}

/* Edge(src,tgt,sd,td): identity is (src, tgt, sd*td) -- min(SHA((s*sd,t*td)), SHA((-s*sd,-t*td))) */
static int32_t edge_get(oracle_graph *g, int32_t src, int32_t tgt, int8_t sd, int8_t td) {
    if ((g->n_edges + 1) * 2 > g->emap_cap && !rehash_edges(g)) return -1;
    int rel = sd * td;
    uint64_t s = edge_hash(src, tgt, rel) & (uint64_t)(g->emap_cap - 1);
    while (g->emap[s] >= 0) {
        int32_t e = g->emap[s];
        if (g->edge_src[e] == src && g->edge_tgt[e] == tgt && g->edge_sd[e] * g->edge_td[e] == rel) return e;
        s = (s + 1) & (uint64_t)(g->emap_cap - 1);
    }
    if (g->n_edges == g->cap_edges) {
        int64_t cap = g->cap_edges ? g->cap_edges * 2 : 4096;
        g->edge_src = realloc(g->edge_src, sizeof(int32_t) * cap);
        g->edge_tgt = realloc(g->edge_tgt, sizeof(int32_t) * cap);
        g->edge_sd = realloc(g->edge_sd, cap);
        g->edge_td = realloc(g->edge_td, cap);
        g->edge_cov = realloc(g->edge_cov, sizeof(uint32_t) * cap);
        if (!g->edge_src || !g->edge_tgt || !g->edge_sd || !g->edge_td || !g->edge_cov) return -1;
        g->cap_edges = cap;
    }
    int32_t e = (int32_t)g->n_edges++;
    g->edge_src[e] = src; g->edge_tgt[e] = tgt; g->edge_sd[e] = sd; g->edge_td[e] = td; g->edge_cov[e] = 0;
    g->emap[s] = e;
    return e;
}

/* canonical form of the k ids at w; returns direction (+1/-1) or 0 for a palindrome */
static int canonical(const int32_t *w, int k, int32_t *out) {
    int dir = 0;
    for (int j = 0; j < k; ++j) {
        int32_t f = w[j], c = -w[k - 1 - j];
        if (f != c) { dir = f < c ? 1 : -1; break; }
    }
    if (dir == 0) return 0;
    if (dir > 0) memcpy(out, w, sizeof(int32_t) * k);
    else for (int j = 0; j < k; ++j) out[j] = -w[k - 1 - j];
    return dir;
}

void oracle_free(oracle_graph *g) {
    if (!g) return;
    free(g->node_key); free(g->node_cov); free(g->node_dir); free(g->node_comp); free(g->node_last_read);
    free(g->map); free(g->inc_node); free(g->inc_read);
    free(g->edge_src); free(g->edge_tgt); free(g->edge_sd); free(g->edge_td); free(g->edge_cov); free(g->emap);
    free(g->win_off); free(g->win_node); free(g->win_dir); free(g->win_start); free(g->win_end);
    free(g->is_short); free(g->to_correct);
    free(g);
}

static uint32_t uf_find(uint32_t *p, uint32_t x) {
    while (p[x] != x) { p[x] = p[p[x]]; x = p[x]; }
    return x;
}

static void label_components(oracle_graph *g) {
    /* ids 1,2,... in order of each component's first node (assign_component_ids) */
    int64_t n = g->n_nodes;
    if (n == 0) return;
    uint32_t *p = malloc(sizeof(uint32_t) * n);
    for (int64_t i = 0; i < n; ++i) p[i] = (uint32_t)i;
    for (int64_t e = 0; e < g->n_edges; ++e) {
        uint32_t a = uf_find(p, (uint32_t)g->edge_src[e]), b = uf_find(p, (uint32_t)g->edge_tgt[e]);
        if (a < b) p[b] = a; else if (b < a) p[a] = b;
    }
    uint32_t next = 0;
    for (int64_t i = 0; i < n; ++i) {
        uint32_t r = uf_find(p, (uint32_t)i);
        if (r == (uint32_t)i) g->node_comp[i] = ++next;       /* root == smallest index in its set */
        else g->node_comp[i] = g->node_comp[r];
    }
    free(p);
}

int oracle_build(oracle_graph **out, const int32_t *ids, const int64_t *off, int64_t R, int32_t k,
                 const int32_t *pos_start, const int32_t *pos_end) {
    *out = NULL;
    if (k < 0 || R < 0) return ORACLE_E_BADARG;
    oracle_graph *g = calloc(1, sizeof(*g));
    if (!g) return ORACLE_E_NOMEM;
    g->k = k; g->R = R;
    g->win_off = calloc(R + 1, sizeof(int64_t));
    g->is_short = calloc(R + 1, 1);
    g->to_correct = calloc(R + 1, 1);
    int64_t W = 0;
    for (int64_t r = 0; r < R; ++r) {
        int64_t L = off[r + 1] - off[r];
        int64_t w = L > k - 1 ? L - (k - 1) : 0;
        if (w && k == 0) { oracle_free(g); return ORACLE_E_BADARG; }   /* GeneMer([]) asserts upstream */
        g->win_off[r] = W;
        g->is_short[r] = w == 0;
        W += w;
    }
    g->win_off[R] = W; g->W = W;
    g->win_node = malloc(sizeof(int32_t) * (W + 1));
    g->win_dir = malloc(W + 1);
    g->win_start = malloc(sizeof(int32_t) * (W + 1));
    g->win_end = malloc(sizeof(int32_t) * (W + 1));
    int32_t *key = malloc(sizeof(int32_t) * (k + 1));
    int rc = ORACLE_OK;
    for (int64_t r = 0; r < R && rc == ORACLE_OK; ++r) {
        int64_t base = off[r], nw = g->win_off[r + 1] - g->win_off[r], w0 = g->win_off[r];
        /* GeneMer construction for every window happens before any insertion (get_geneMers) */
        for (int64_t i = 0; i < nw; ++i) {
            int d = canonical(ids + base + i, k, key);
            if (d == 0) { rc = ORACLE_E_PALINDROME; break; }
            g->win_dir[w0 + i] = (int8_t)d;
        }
        if (rc != ORACLE_OK) break;
        int32_t prev = -1;
        for (int64_t i = 0; i < nw; ++i) {
            int32_t n;
            if (i == 0) {
                canonical(ids + base, k, key);
                n = node_get(g, key, g->win_dir[w0]);
            } else n = prev;
            if (n < 0 || !node_touch(g, n, (int32_t)r)) { rc = ORACLE_E_NOMEM; break; }
            g->win_node[w0 + i] = n;
            g->win_start[w0 + i] = pos_start ? pos_start[base + i] : -1;
            g->win_end[w0 + i] = pos_end ? pos_end[base + i + k - 1] : -1;
            g->node_cov[n] += 1;
            if (i + 1 < nw) {
                canonical(ids + base + i + 1, k, key);
                int32_t t = node_get(g, key, g->win_dir[w0 + i + 1]);
                if (t < 0 || !node_touch(g, t, (int32_t)r)) { rc = ORACLE_E_NOMEM; break; }
                int8_t sd = g->win_dir[w0 + i], td = g->win_dir[w0 + i + 1];
                int32_t fwd = edge_get(g, n, t, sd, td);
                int32_t rev = edge_get(g, t, n, (int8_t)-td, (int8_t)-sd);
                if (fwd < 0 || rev < 0) { rc = ORACLE_E_NOMEM; break; }
                g->edge_cov[fwd] += 1;
                g->edge_cov[rev] += 1;
                prev = t;
            }
        }
    }
    free(key);
    if (rc != ORACLE_OK) { oracle_free(g); return rc; }
    label_components(g);
    *out = g;
    return ORACLE_OK;
}

/* remove flagged nodes (and every edge touching them), and flagged edges; preserves orders */
static void apply_removal(oracle_graph *g, const uint8_t *node_rm, uint8_t *edge_rm) {
    int64_t n = g->n_nodes, m = g->n_edges;
    int32_t *remap = malloc(sizeof(int32_t) * (n + 1));
    for (int64_t e = 0; e < m; ++e)
        if (node_rm[g->edge_src[e]] || node_rm[g->edge_tgt[e]]) edge_rm[e] = 1;
    int64_t nn = 0;
    for (int64_t i = 0; i < n; ++i) {
        if (node_rm[i]) { remap[i] = -1; continue; }
        remap[i] = (int32_t)nn;
        if (nn != i) {
            memmove(g->node_key + nn * g->k, g->node_key + i * g->k, sizeof(int32_t) * g->k);
            g->node_cov[nn] = g->node_cov[i]; g->node_dir[nn] = g->node_dir[i]; g->node_comp[nn] = g->node_comp[i];
        }
        nn++;
    }
    /* remove_node_from_reads: every read on a removed node is marked, its windows become None */
    int64_t ni = 0;
    for (int64_t i = 0; i < g->n_inc; ++i) {
        if (node_rm[g->inc_node[i]]) { g->to_correct[g->inc_read[i]] = 1; continue; }
        g->inc_node[ni] = remap[g->inc_node[i]]; g->inc_read[ni] = g->inc_read[i]; ni++;
    }
    g->n_inc = ni;
    for (int64_t w = 0; w < g->W; ++w) {
        int32_t x = g->win_node[w];
        if (x < 0) continue;
        if (node_rm[x]) { g->win_node[w] = -1; g->win_dir[w] = 0; g->win_start[w] = -1; g->win_end[w] = -1; }
        else g->win_node[w] = remap[x];
    }
    int64_t mm = 0;
    for (int64_t e = 0; e < m; ++e) {
        if (edge_rm[e]) continue;
        g->edge_src[mm] = remap[g->edge_src[e]]; g->edge_tgt[mm] = remap[g->edge_tgt[e]];
        g->edge_sd[mm] = g->edge_sd[e]; g->edge_td[mm] = g->edge_td[e]; g->edge_cov[mm] = g->edge_cov[e];
        mm++;
    }
    g->n_nodes = nn; g->n_edges = mm;
    free(remap);
    /* the lookup maps are only needed during the build */
    free(g->map); g->map = NULL; g->map_cap = 0;
    free(g->emap); g->emap = NULL; g->emap_cap = 0;
}

int oracle_filter(oracle_graph *g, uint32_t min_node_cov, uint32_t min_edge_cov) {
    uint8_t *nrm = calloc(g->n_nodes + 1, 1), *erm = calloc(g->n_edges + 1, 1);
    for (int64_t i = 0; i < g->n_nodes; ++i) nrm[i] = g->node_cov[i] < min_node_cov;
    for (int64_t e = 0; e < g->n_edges; ++e) erm[e] = g->edge_cov[e] < min_edge_cov;
    apply_removal(g, nrm, erm);
    free(nrm); free(erm);
    return ORACLE_OK;
}

/* remove_node -> get_edge_hashes_between_nodes returns lists when a doomed node has two edges
   to the same neighbour; upstream then raises TypeError.  Only possible for k = 1 / even k.
   Two edges between the same ordered pair always differ in relative orientation (sd * td). */
static int has_multi_edge(oracle_graph *g, const uint8_t *node_rm) {
    if (!g->emap) {  /* dropped by an earlier removal: rebuild it at its final size (a full table never ends a probe) */
        int64_t cap = 4096;
        while (cap < 2 * g->n_edges + 2) cap *= 2;
        g->emap_cap = cap / 2;
        rehash_edges(g);
    }
    for (int64_t e = 0; e < g->n_edges; ++e) {
        if (!node_rm[g->edge_src[e]]) continue;
        int rel = -(g->edge_sd[e] * g->edge_td[e]);
        uint64_t s = edge_hash(g->edge_src[e], g->edge_tgt[e], rel) & (uint64_t)(g->emap_cap - 1);
        while (g->emap[s] >= 0) {
            int32_t f = g->emap[s];
            if (g->edge_src[f] == g->edge_src[e] && g->edge_tgt[f] == g->edge_tgt[e] &&
                g->edge_sd[f] * g->edge_td[f] == rel) return 1;
            s = (s + 1) & (uint64_t)(g->emap_cap - 1);
        }
    }
    return 0;
}

int oracle_remove_low_coverage_components(oracle_graph *g, uint32_t min_component_cov) {
    uint32_t maxc = 0;
    for (int64_t i = 0; i < g->n_nodes; ++i) if (g->node_comp[i] > maxc) maxc = g->node_comp[i];
    uint32_t *best = calloc((size_t)maxc + 1, sizeof(uint32_t));
    for (int64_t i = 0; i < g->n_nodes; ++i)
        if (g->node_cov[i] > best[g->node_comp[i]]) best[g->node_comp[i]] = g->node_cov[i];
    uint8_t *nrm = calloc(g->n_nodes + 1, 1), *erm = calloc(g->n_edges + 1, 1);
    for (int64_t i = 0; i < g->n_nodes; ++i) nrm[i] = best[g->node_comp[i]] < min_component_cov;
    free(best);
    if (has_multi_edge(g, nrm)) { free(nrm); free(erm); return ORACLE_E_MULTIEDGE; }
    apply_removal(g, nrm, erm);
    free(nrm); free(erm);
    return ORACLE_OK;
}

/* remove_node (construct_graph.py:463-484) for every node whose flag is set; nothing changes on a multi-edge */
int oracle_remove_nodes(oracle_graph *g, const uint8_t *flags) {
    uint8_t *nrm = calloc(g->n_nodes + 1, 1), *erm = calloc(g->n_edges + 1, 1);
    for (int64_t i = 0; i < g->n_nodes; ++i) nrm[i] = flags[i] != 0;
    if (has_multi_edge(g, nrm)) { free(nrm); free(erm); return ORACLE_E_MULTIEDGE; }
    apply_removal(g, nrm, erm);
    free(nrm); free(erm);
    return ORACLE_OK;
}

void oracle_sizes(const oracle_graph *g, int64_t *n_nodes, int64_t *n_edges, int64_t *n_windows,
                  int64_t *n_incidence, int64_t *n_fw, int64_t *n_bw) {
    int64_t fw = 0, bw = 0;
    for (int64_t e = 0; e < g->n_edges; ++e) { if (g->edge_sd[e] > 0) fw++; else bw++; }
    *n_nodes = g->n_nodes; *n_edges = g->n_edges; *n_windows = g->W; *n_incidence = g->n_inc; *n_fw = fw; *n_bw = bw;
}

void oracle_export_nodes(const oracle_graph *g, int32_t *key, uint32_t *cov, int8_t *first_dir, uint32_t *component,
                         int64_t *reads_off, int32_t *reads, int64_t *fw_off, int32_t *fw_edges,
                         int64_t *bw_off, int32_t *bw_edges) {
    int64_t n = g->n_nodes;
    memcpy(key, g->node_key, sizeof(int32_t) * n * g->k);
    memcpy(cov, g->node_cov, sizeof(uint32_t) * n);
    memcpy(first_dir, g->node_dir, n);
    memcpy(component, g->node_comp, sizeof(uint32_t) * n);
    /* stable counting sort of the incidence events by node keeps reads ascending */
    memset(reads_off, 0, sizeof(int64_t) * (n + 1));
    for (int64_t i = 0; i < g->n_inc; ++i) reads_off[g->inc_node[i] + 1]++;
    for (int64_t i = 0; i < n; ++i) reads_off[i + 1] += reads_off[i];
    int64_t *cur = malloc(sizeof(int64_t) * (n + 1));
    memcpy(cur, reads_off, sizeof(int64_t) * (n + 1));
    for (int64_t i = 0; i < g->n_inc; ++i) reads[cur[g->inc_node[i]]++] = g->inc_read[i];
    /* an edge sits in its source node's forward list iff its stored source direction is +1
       (add_edge_to_node, construct_graph.py:287-298); list order = edge creation order */
    memset(fw_off, 0, sizeof(int64_t) * (n + 1));
    memset(bw_off, 0, sizeof(int64_t) * (n + 1));
    for (int64_t e = 0; e < g->n_edges; ++e) (g->edge_sd[e] > 0 ? fw_off : bw_off)[g->edge_src[e] + 1]++;
    for (int64_t i = 0; i < n; ++i) { fw_off[i + 1] += fw_off[i]; bw_off[i + 1] += bw_off[i]; }
    memcpy(cur, fw_off, sizeof(int64_t) * (n + 1));
    for (int64_t e = 0; e < g->n_edges; ++e) if (g->edge_sd[e] > 0) fw_edges[cur[g->edge_src[e]]++] = (int32_t)e;
    memcpy(cur, bw_off, sizeof(int64_t) * (n + 1));
    for (int64_t e = 0; e < g->n_edges; ++e) if (g->edge_sd[e] < 0) bw_edges[cur[g->edge_src[e]]++] = (int32_t)e;
    free(cur);
}

void oracle_export_edges(const oracle_graph *g, int32_t *src, int32_t *tgt, int8_t *sd, int8_t *td, uint32_t *cov) {
    int64_t m = g->n_edges;
    memcpy(src, g->edge_src, sizeof(int32_t) * m); memcpy(tgt, g->edge_tgt, sizeof(int32_t) * m);
    memcpy(sd, g->edge_sd, m); memcpy(td, g->edge_td, m); memcpy(cov, g->edge_cov, sizeof(uint32_t) * m);
}

void oracle_export_reads(const oracle_graph *g, int64_t *win_off, int32_t *node_idx, int8_t *dir, int32_t *start,
                         int32_t *end, uint8_t *is_short, uint8_t *to_correct) {
    memcpy(win_off, g->win_off, sizeof(int64_t) * (g->R + 1));
    memcpy(node_idx, g->win_node, sizeof(int32_t) * g->W);
    memcpy(dir, g->win_dir, g->W);
    if (start) memcpy(start, g->win_start, sizeof(int32_t) * g->W);
    if (end) memcpy(end, g->win_end, sizeof(int32_t) * g->W);
    memcpy(is_short, g->is_short, g->R);
    memcpy(to_correct, g->to_correct, g->R);
}
