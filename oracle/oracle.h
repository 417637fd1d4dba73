/*
 * oracle/oracle.h -- TEST INFRASTRUCTURE: CPU restatement of the hot path.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load this library; the product (embiggen_b200/)
 * never does.
 *
 * PARITY UNPINNED against Ensmallen: the reference's arithmetic for this path
 * lives in the third-party Rust wheel `ensmallen>=0.8.94`
 * (/root/reference/setup.py:76, call site
 * /root/reference/embiggen/embedders/ensmallen_embedders/node2vec.py:99) whose
 * source is not vendored and which no reference test pins numerically
 * (SURVEY.md 8c).  What this oracle IS pinned against:
 *   - Random123 known-answer vectors for Philox4x32-10,
 *   - the analytic node2vec transition pmf (Grover & Leskovec 2016, eq. 2)
 *     by chi-square on small graphs,
 *   - the target pmf deg^alpha for the alias table,
 *   - an independent numpy restatement of the SkipGram/CBOW update
 *     (tests/test_oracle_sgns.py) and committed fixtures in tests/golden/.
 * Semantics of every kwarg follow the reference docstrings
 * /root/reference/embiggen/embedders/ensmallen_embedders/node2vec_skipgram.py:37-119.
 */
#ifndef ORACLE_H
#define ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORC_PAD_TOKEN 0xFFFFFFFFu
#define ORC_MAX_TRIALS (1u << 20)

typedef struct {
    uint64_t steps;          /* sampled transitions                                        */
    uint64_t trials;         /* proposals drawn by second-order steps                      */
    uint64_t first_order;    /* steps taken with the uniform (first-order) rule            */
    uint64_t searches;       /* adjacency checks not resolved by return / bound shortcuts  */
    uint64_t probe_sectors;  /* 32 B sectors those checks touch (SURVEY.md 8d S_probe)     */
    uint64_t capped;         /* steps that hit ORC_MAX_TRIALS                              */
} orc_walk_counters;

/* Philox4x32-10, key = (seed lo, seed hi); exported for the known-answer tests */
void orc_philox(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]);

/* nodes with degree > 0, ascending; returns their count (out may be NULL). */
uint64_t orc_sources(const int64_t *indptr, uint64_t n, uint32_t *out);

/* thresholds of the integer accept test, SURVEY.md App. C.4 */
void orc_thresholds(float return_weight, float explore_weight, uint64_t thr[3]);

/*
 * Walk ids are first_walk + i * walk_id_stride, i in [0, n_walks); walk id g
 * starts at sources[g % n_src].  out is row-major [n_walks][walk_length].
 */
int orc_walks(const int64_t *indptr, const uint32_t *indices, uint64_t n, const uint32_t *sources,
              uint64_t n_src, uint64_t seed, uint64_t first_walk, uint64_t n_walks,
              uint64_t walk_id_stride, uint32_t walk_length, float return_weight,
              float explore_weight, int undirected, uint32_t *out, orc_walk_counters *counters);

/* `undirected` (every edge has its mirror; orc_is_undirected) lets the sampler fold the return
 * edge out of the rejection envelope when return_weight > max(1, explore_weight): walks.c */
int orc_is_undirected(const int64_t *indptr, const uint32_t *indices, uint64_t n);
void orc_fold_thresholds(float return_weight, float explore_weight, uint64_t thrf[3], uint64_t *excess);

/* per-row alias tables of a weighted graph (see walks.c): two words per edge, {thr, alias index
 * inside the row}.  The `table` arguments below take this table (NULL: unweighted). */
int orc_edge_alias(const int64_t *indptr, const float *weights, uint64_t n, uint32_t *table);

/* orc_walks with proposals proportional to the edge weights (table from orc_edge_alias; NULL: uniform) */
int orc_walks_weighted(const int64_t *indptr, const uint32_t *indices, const uint32_t *table, uint64_t n,
                       const uint32_t *sources, uint64_t n_src, uint64_t seed, uint64_t first_walk,
                       uint64_t n_walks, uint64_t walk_id_stride, uint32_t walk_length,
                       float return_weight, float explore_weight, int undirected, uint32_t *out,
                       orc_walk_counters *counters);

/* orc_walks_weighted plus typed walks: node_types[n] / edge_types[nnz] (NULL: untyped) and the
 * weights multiplied in when the node type / the edge type changes.  normalize_by_degree is a
 * property of the proposal table: build `table` over weight / max(deg(destination), 1). */
void orc_type_thresholds(float change_weight, uint64_t q[2]);
int orc_walks_typed(const int64_t *indptr, const uint32_t *indices, const uint32_t *table,
                    const uint32_t *node_types, const uint32_t *edge_types,
                    float change_node_type_weight, float change_edge_type_weight, uint64_t n,
                    const uint32_t *sources, uint64_t n_src, uint64_t seed, uint64_t first_walk,
                    uint64_t n_walks, uint64_t walk_id_stride, uint32_t walk_length,
                    float return_weight, float explore_weight, int undirected, uint32_t *out,
                    orc_walk_counters *counters);

/* Alias table over deg^alpha (integer construction, alias.c); thr/alias have n entries. */
int orc_alias_fraction_bits(uint64_t n, uint64_t max_degree, double alpha);
int orc_alias_build(const int64_t *indptr, uint64_t n, double alpha, uint32_t *thr,
                    uint32_t *alias);

typedef struct {
    uint32_t model; /* 0 SkipGram, 1 CBOW */
    uint32_t embedding_size;
    uint32_t row_stride; /* floats per row, multiple of 4, >= embedding_size */
    uint32_t walk_length;
    uint32_t window_size;
    uint32_t negatives;
    float clipping_value;
    float learning_rate;
    uint32_t use_alias;                         /* 0 => uniform negatives                   */
    uint32_t normalize_learning_rate_by_degree; /* lr / deg(centre)                         */
    uint32_t scale_by_sqrt_dim;                 /* dot / sqrt(D)  (P, SURVEY.md App. C.6)   */
    uint32_t downsample_bound; /* stochastic_downsample_by_degree: max degree + 1, 0 => off */
    uint32_t fast_math; /* 1: vectorised dot + libm expf: for timing the CPU baseline only (sgns.c) */
    uint32_t shared_negatives; /* SkipGram only, opt-in: one set of negatives per CENTRE, shared by
                                  its pairs (north_star's shared-negative batching; sgns.c)        */
} orc_sgns_cfg;

/*
 * threads > 1 turns orc_walks / orc_train into OpenMP loops over walks
 * (Hogwild for the tables, like the reference engine's rayon pool).  Used
 * only to time the CPU baseline; parity tests run with 1 (the default).
 */
void orc_set_threads(int threads);
int orc_get_threads(void);

void orc_philox_range(uint64_t seed, uint32_t first_c0, uint64_t count, uint32_t c1, uint32_t c2,
                      uint32_t c3, uint32_t *out);
float orc_exp_det(float y); /* exp from IEEE single ops only (Cody-Waite + degree-6 polynomial) */
float orc_log_det(float x); /* ln  from IEEE single ops only (atanh series), x > 0, normal      */
float orc_sigmoid(float x);
float orc_dot(const float *a, const float *b, uint32_t row_stride);

int orc_init_tables(uint64_t n, uint32_t embedding_size, uint32_t row_stride, uint64_t seed,
                    float *t0, float *t1);

/*
 * Seeded synthetic graphs of the BASELINE.json shapes (graphgen.c): the first n_edges distinct
 * undirected edges, in draw order, of the Philox stream (seed, draw index); kind 0 = Erdos-Renyi
 * G(n, m), kind 1 = R-MAT over 2^scale ids with ids >= n rejected and quadrant thresholds
 * t_a, t_ab, t_abc (floor(p * 2^32)).  indptr has n + 1 entries, indices 2 * n_edges.  Same graph
 * as embiggen_b200/graph.py (numpy) and the product's GPU builder; OpenMP over orc_set_threads.
 */
int orc_synthetic_csr(int kind, uint64_t n, uint32_t scale, uint64_t n_edges, uint64_t seed, uint64_t t_a,
                      uint64_t t_ab, uint64_t t_abc, int64_t *indptr, uint32_t *indices, uint64_t *nnz_out);

/*
 * Sequential deterministic training over row-major walks (ascending order).
 * loss_sum / pairs / targets are accumulated into (may be NULL).
 */
int orc_train(const orc_sgns_cfg *cfg, const uint32_t *walks, uint64_t n_walks,
              uint64_t first_walk, uint64_t walk_id_stride, uint64_t seed, uint64_t n,
              const int64_t *indptr, const uint32_t *thr, const uint32_t *alias, float *t0,
              float *t1, double *loss_sum, uint64_t *pairs, uint64_t *targets);

/*
 * GloVe on the walk co-occurrences ("next" row f-3; wrappers
 * /root/reference/embiggen/embedders/ensmallen_embedders/node2vec_glove.py:5-140,
 * deepwalk_glove.py).  Triples (centre, context, count) sorted by (centre, context); per centre
 * the row of T0 stays in `h` while its contexts are visited in order:
 *   f = <h, T1[o]>;  skipped when |f| > clipping_value
 *   weight = exp(alpha * ln(count / max_count));  g = 2 * weight * (f - ln(count)) * lr
 *   h' = h - g * T1[o];  T1[o] -= g * h;  h = h'
 * loss_sum accumulates weight * (f - ln count)^2 over the triples that were not skipped.
 *
 * tile_semantics != 0 restates the arithmetic of the production GPU kernel (glove.cu:
 * glove_tile_kernel) instead of the specification above, for runs of one centre that no tile
 * boundary splits: the context row takes T1[o] + (-g * h) rounded twice (a product, then an
 * atomic add) instead of one fused multiply-add, and the centre row is written back as
 * T0[c] + (h - h0), h0 being the row as the run loaded it, instead of h.
 */
int orc_glove_train(const uint32_t *centre, const uint32_t *context, const uint32_t *count,
                    uint64_t n_triples, uint32_t max_count, uint32_t embedding_size,
                    uint32_t row_stride, float alpha, float clipping_value, float learning_rate,
                    int tile_semantics, float *t0, float *t1, double *loss_sum, uint64_t *trained);

#ifdef __cplusplus
}
#endif
#endif
