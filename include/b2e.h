/*
 * include/b2e.h -- C ABI of the B200-native Node2Vec/DeepWalk SkipGram & CBOW engine.
 *
 * This is the drop-in boundary for ONE path of monarch-initiative/embiggen: what
 * `ensmallen.models.SkipGram / CBOW` do below the PyO3 call at
 * /root/reference/embiggen/embedders/ensmallen_embedders/node2vec.py:99
 * (`self._model.fit_transform(graph)`), constructed at node2vec.py:65-69 from the
 * kwargs declared in .../node2vec_skipgram.py:9-146.  The reference's own FFI is PyO3
 * (process-internal, Rust objects); a replacement binds these entry points instead
 * (ctypes stub in INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a
 * negative b2e_status, never aborts; b2e_last_error() gives the thread-local message the
 * Python shim turns into ValueError / RuntimeError (reference error behaviour:
 * .../abstract_embedding_model.py:114-166).  The caller owns host buffers; the library
 * owns device memory for the lifetime of a handle.  There is no CPU fallback: without a
 * CUDA device b2e_create fails with B2E_ERR_CUDA.
 */
#ifndef B2E_H
#define B2E_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2E_ABI_VERSION 3
#define B2E_PAD_TOKEN 0xFFFFFFFFu /* walk token after a dead end (directed graphs only) */
#define B2E_MAX_WORLD 16          /* replicas one exchange step can average (GPUs of one node) */
#define B2E_IPC_HANDLE_BYTES 64   /* sizeof(cudaIpcMemHandle_t) */

typedef enum {
    B2E_OK = 0,
    B2E_ERR_INVALID = -1, /* bad argument / unsupported configuration */
    B2E_ERR_CUDA = -2,    /* CUDA runtime failure, device missing, out of memory */
    B2E_ERR_STATE = -3    /* call order violated (e.g. fit before load_csr) */
} b2e_status;

typedef enum { B2E_SKIPGRAM = 0, B2E_CBOW = 1, B2E_GLOVE = 2 } b2e_model;

/*
 * Mirrors the constructor kwargs of Node2VecSkipGramEnsmallen / Node2VecCBOWEnsmallen
 * (.../node2vec_skipgram.py:9-35, node2vec_cbow.py) that reach the native engine.
 * DeepWalk = return_weight == explore_weight == 1 (.../deepwalk_skipgram.py:6-139).
 */
typedef struct {
    uint32_t struct_size; /* sizeof(b2e_config), ABI check */
    uint32_t model;       /* b2e_model */
    uint32_t embedding_size;
    uint32_t epochs;
    uint32_t walk_length;
    uint32_t iterations;
    uint32_t window_size;
    uint32_t number_of_negative_samples;
    float clipping_value;
    float return_weight;  /* 1/p */
    float explore_weight; /* 1/q */
    float learning_rate;
    float learning_rate_decay;
    float negative_sampling_exponent;           /* alias table over deg^alpha; north_star: 0.75 */
    float glove_alpha;             /* GloVe: weight (count / max count)^alpha (node2vec_glove.py:37) */
    float change_node_type_weight; /* walk weight x this when the node type changes (b2e_load_types) */
    float change_edge_type_weight; /* ... when the edge type changes; 1 = untyped walks */
    uint32_t use_scale_free_distribution;       /* 0 => uniform negatives */
    uint32_t normalize_learning_rate_by_degree; /* lr / deg(centre) */
    uint32_t normalize_by_degree;               /* walk transition weight / deg(destination) */
    uint32_t stochastic_downsample_by_degree;   /* skip a centre with probability deg / (max deg + 1) */
    uint32_t scale_by_sqrt_dim;                 /* score = dot / sqrt(D) */
    uint32_t walklet_scale; /* k >= 2: Walklets (.../walklets.py), train on the k sub-walks made of
                               every k-th token, so that `window_size` counts in hops of k */
    uint32_t shared_negatives; /* SkipGram, opt-in (north_star's shared-negative batching): one set of
                                  negatives per CENTRE, shared by its pairs, each negative weighted by
                                  the number of pairs it stands for; needs window_size <= 7,
                                  number_of_negative_samples <= 15, embedding_size <= 128 */
    uint32_t deterministic; /* 1: one warp trains walks in ascending id order (bit-exact) */
    uint32_t chunk_walks;   /* walks per walk->SGD chunk, 0 = automatic */
    uint32_t max_concurrent_walks; /* walks trained concurrently (Hogwild), 0 = automatic */
    int32_t device;         /* CUDA device ordinal */
} b2e_config;

/* Event counters accumulated on the device (roofline accounting, SURVEY.md 8d). */
typedef struct {
    uint64_t walk_steps;    /* sampled transitions */
    uint64_t walk_trials;   /* second-order proposals */
    uint64_t walk_searches; /* adjacency checks the accept test could not decide without the class */
    uint64_t walk_probes;   /* gathers those checks cost: row-filter words, row bounds, bisection steps */
    uint64_t walk_filter_rejects; /* checks answered "not a neighbour" by the row filter alone */
    uint64_t pairs;         /* (centre, context) positives trained */
    uint64_t targets;       /* target rows scored (positive + valid negatives) */
    double loss_sum;        /* sum of pair losses since the last b2e_reset_counters */
} b2e_counters;

typedef struct b2e_handle b2e_handle;

const char *b2e_last_error(void);
int b2e_abi_version(void);
/* number of visible devices this library can run on (compute capability >= 10.0); 0 if none */
int b2e_device_count(void);
/* Make `device` the current CUDA device of the calling thread.  The handle-free entry points
 * (b2e_edge_metrics, b2e_perceptron_fit / _predict without node features, the graph builders)
 * run on the current device; handles and feature matrices carry their own. */
int b2e_select_device(int device);

int b2e_create(const b2e_config *config, b2e_handle **out);
void b2e_destroy(b2e_handle *handle);

/*
 * K1: copy GRAPE's sorted neighbour arrays into HBM once.  indptr has n + 1 entries
 * (0 followed by get_cumulative_node_degrees(), .../pecanpy_embedders/node2vec.py:144-148),
 * indices has nnz sorted-per-row destination ids (get_directed_destination_node_ids(), :161).
 * Host pointers.  Also derives the start-node list (degree > 0) and the alias table (K3).
 */
int b2e_load_csr(b2e_handle *handle, const int64_t *indptr, const uint32_t *indices,
                 uint64_t n, uint64_t nnz);

/*
 * Same with edge weights (get_directed_edge_weights(), .../pecanpy_embedders/node2vec.py:147):
 * nnz non-negative float32 aligned with indices; proposals are drawn proportionally to them
 * (the reference's classes are `is_using_edge_weights`, .../ensmallen_embedders/node2vec.py:119-129).
 * weights == NULL is b2e_load_csr.
 */
int b2e_load_csr_weighted(b2e_handle *handle, const int64_t *indptr, const uint32_t *indices,
                          const float *weights, uint64_t n, uint64_t nnz);

/*
 * Typed walks: the type ids behind `change_node_type_weight` / `change_edge_type_weight`
 * (.../node2vec_skipgram.py:72-77; the reference reads them from the graph:
 * `graph.get_single_label_node_type_ids()`, `graph.get_directed_edge_type_ids()`).  node_types
 * has n entries, edge_types nnz entries in CSR order; either may be NULL.  Call after
 * b2e_load_csr* (which drops the types of the previous graph); a change weight whose types were
 * never loaded has no effect (the graph walks untyped).
 */
int b2e_load_types(b2e_handle *handle, const uint32_t *node_types, const uint32_t *edge_types);

/*
 * GloVe (model B2E_GLOVE; replaces `ensmallen.models.GloVe.fit_transform` behind
 * node2vec_glove.py / deepwalk_glove.py).  b2e_fit runs the whole path; the pieces, for parity
 * tests: b2e_cooccurrence walks `n_walks` walks and counts the ordered pairs of different
 * tokens at most `window_size` apart (accumulate != 0 adds to the resident counts instead of
 * replacing them); b2e_cooccurrence_export copies the triples, sorted by (centre, context);
 * b2e_glove_train is one pass of SGD over the resident triples (counters: pairs = triples
 * trained, loss_sum = sum of weight * (dot - ln count)^2).
 */
int b2e_cooccurrence(b2e_handle *handle, uint64_t seed, uint64_t first_walk, uint64_t n_walks,
                     uint64_t walk_id_stride, int accumulate, uint64_t *n_triples);
int b2e_cooccurrence_export(b2e_handle *handle, uint32_t *centre, uint32_t *context, uint32_t *count);
int b2e_glove_train(b2e_handle *handle, float learning_rate);

/*
 * GloVe on several GPUs: the centre ids are sharded over the ranks, the tables merged once per
 * epoch (csrc/exchange.cu; normative statement: oracle.glove_fit_sharded).  Per epoch, on every rank:
 *   b2e_glove_walk_epoch   walks the whole epoch (ids first_walk .. first_walk + n_walks - 1) into
 *                          HBM and takes its token histogram; identical on every rank;
 *   b2e_glove_shard_count  splits [0, n) into `world` intervals of centre id balanced by key slots
 *                          (owner_bounds, may be NULL, receives world + 1 entries: rank r owns
 *                          [owner_bounds[r], owner_bounds[r + 1])) and counts this rank's centres,
 *                          range by range within the sort capacity; *local_max receives their
 *                          largest count (0 if none);
 *   b2e_glove_shard_train  one SGD pass over this rank's centres in ascending order, weights against
 *                          max_count, the largest count of the whole epoch (the maximum of the ranks'
 *                          local_max); with world > 1 it first snapshots T1 on the device;
 *   b2e_glove_merge        asynchronous on the train stream, over the peers of b2e_exchange_open*:
 *                          every replica takes row v of T0 from the owner of v, and T1 becomes
 *                          snapshot + sum over the ranks of (T1_rank - snapshot); bracketed by
 *                          barriers like b2e_exchange_average.  Afterwards the replicas are
 *                          bit-identical.  A no-op with world 1.
 */
int b2e_glove_walk_epoch(b2e_handle *handle, uint64_t seed, uint64_t first_walk, uint64_t n_walks);
int b2e_glove_shard_count(b2e_handle *handle, uint32_t world, uint32_t rank, uint32_t *owner_bounds,
                          uint32_t *local_max);
int b2e_glove_shard_train(b2e_handle *handle, float learning_rate, uint32_t max_count);
int b2e_glove_merge(b2e_handle *handle);

uint64_t b2e_number_of_sources(const b2e_handle *handle);
uint64_t b2e_row_stride(const b2e_handle *handle); /* floats per table row on the device */

/*
 * The whole path, host buffers in and out: replaces `model.fit_transform(graph)`
 * (node2vec.py:99).  table0 / table1 receive n x embedding_size float32, row-major, in
 * [central, contextual] role order like the reference; epoch_loss (may be NULL) receives
 * `epochs` mean pair losses.  The seed is read here, not at create time (SURVEY.md 8b).
 */
int b2e_fit(b2e_handle *handle, uint64_t seed, float *table0, float *table1, float *epoch_loss);

/*
 * K2, parity/debug export: walks with ids first_walk + i * walk_id_stride, i < n_walks,
 * row-major [n_walks][walk_length] uint32 into a host buffer.
 */
int b2e_walks(b2e_handle *handle, uint64_t seed, uint64_t first_walk, uint64_t n_walks,
              uint64_t walk_id_stride, uint32_t *out);

/*
 * The first n_walks walks of a walk slot as the last b2e_walk_chunk / b2e_train_host_walks left
 * them (what b2e_train_chunk on that slot consumes), row-major [n_walks][walk_length] uint32
 * into a host buffer.  Not for Walklets, whose slots hold the split walks.
 */
int b2e_slot_walks(b2e_handle *handle, uint32_t slot, uint64_t n_walks, uint32_t *out);

/*
 * Page-lock / unlock a caller-owned host buffer (cudaHostRegister): b2e_fit then copies the tables
 * of a large graph into it at full PCIe speed (40 GB per table at 100 M nodes).  Optional.
 */
int b2e_host_register(void *buffer, uint64_t bytes);
int b2e_host_unregister(void *buffer);

/* ---- stepping API (device-resident; used by the host driver, multi-GPU and bench) ---- */

/* Streams are cudaStream_t handles (e.g. torch.cuda.Stream().cuda_stream); NULL = default. */
int b2e_set_streams(b2e_handle *handle, void *walk_stream, void *train_stream);
int b2e_init_tables(b2e_handle *handle, uint64_t seed);
/* walks for one chunk into device buffer `slot` (0 or 1), asynchronous on the walk stream */
int b2e_walk_chunk(b2e_handle *handle, uint64_t seed, uint64_t first_walk, uint64_t n_walks,
                   uint64_t walk_id_stride, uint32_t slot);
/* Walklets in one pass (.../walklets.py:7-149: one embedding per scale): `handle` takes the chunk
 * `source` has just walked into `slot` (split by handle's own walklet_scale) instead of walking it
 * again; the source must not walk into that slot again before its adopters have trained on it */
int b2e_adopt_walks(b2e_handle *handle, b2e_handle *source, uint32_t slot);
/* K4/K5 over the walks in `slot`, asynchronous on the train stream, ordered after the walk */
int b2e_train_chunk(b2e_handle *handle, uint64_t seed, uint32_t slot, float learning_rate);
/* train on caller-provided host walks (parity tests feed the oracle's walks) */
int b2e_train_host_walks(b2e_handle *handle, uint64_t seed, const uint32_t *walks,
                         uint64_t first_walk, uint64_t n_walks, uint64_t walk_id_stride,
                         float learning_rate);
int b2e_sync(b2e_handle *handle);

/* device pointers of the two tables (n x row_stride float32) */
int b2e_device_tables(b2e_handle *handle, void **table0, void **table1);

/*
 * The exchange step of the data-parallel path (north_star subsystem 4; no counterpart in the
 * reference, whose engine is one shared-memory process): every GPU of the node holds a replica of
 * both tables, trains its shard of the walks on it, and the replicas are averaged at a fixed step
 * interval.  One kernel per rank reduces the rows that rank owns over NVLink peer memory and
 * writes the average back to every replica (csrc/exchange.cu).
 *   b2e_exchange_handles   writes the CUDA IPC handles of this replica's two tables
 *                          (2 x B2E_IPC_HANDLE_BYTES) for the other processes of the node;
 *   b2e_exchange_open      takes the handles of all `world` ranks, rank-major (this rank's own
 *                          entry is ignored), and maps the peers' tables;
 *   b2e_exchange_open_local same with replicas that live in this process (handles[world], tests);
 *   b2e_exchange_average   asynchronous on the train stream; the caller guarantees that every
 *                          replica has finished its SGD chunk before any rank starts (barrier) and
 *                          that no rank resumes before all have finished (second barrier);
 *   b2e_exchange_close     unmaps the peers (also done by b2e_load_csr* and b2e_destroy).
 * b2e_tables_digest: {sum, sum of squares} of table 0, of table 1 (4 doubles), then the
 * wrap-around sums of the float bit patterns of the two tables and the number of non-finite values
 * (3 uint64): equal replicas give equal words.
 */
int b2e_exchange_handles(b2e_handle *handle, void *ipc_handles);
int b2e_exchange_open(b2e_handle *handle, uint32_t world, uint32_t rank, const void *all_ipc_handles);
int b2e_exchange_open_local(b2e_handle *handle, uint32_t world, uint32_t rank, b2e_handle *const *replicas);
int b2e_exchange_average(b2e_handle *handle);
int b2e_exchange_close(b2e_handle *handle);
int b2e_tables_digest(b2e_handle *handle, double *sums, uint64_t *words);
int b2e_chunk_capacity(const b2e_handle *handle, uint64_t *walks);
/* strip the row padding and copy both tables to host buffers (n x embedding_size each) */
int b2e_export_tables(b2e_handle *handle, float *table0, float *table1);
/* overwrite both device tables from host buffers (n x embedding_size each) */
int b2e_import_tables(b2e_handle *handle, const float *table0, const float *table1);
/* alias table as built for the handle (n entries each); parity/debug export */
int b2e_export_alias(b2e_handle *handle, uint32_t *threshold, uint32_t *alias);
/* per-row alias tables of a weighted load (nnz x 2 words: {thr, alias index inside the row}, the
 * layout of oracle/walks.c: orc_edge_alias), as built on the device; parity/debug export.
 * B2E_ERR_STATE when the handle walks without weights. */
int b2e_export_edge_alias(b2e_handle *handle, uint32_t *table);

int b2e_counters_read(b2e_handle *handle, b2e_counters *out);
int b2e_counters_reset(b2e_handle *handle);
/* number of kernels this handle has launched since creation */
uint64_t b2e_launch_count(const b2e_handle *handle);

/* ---- graph ingest on the GPU (SURVEY.md 8(f) row 1; no handle needed) ---- */

/*
 * Sorted, de-duplicated, self-loop-free CSR from a host edge list: the layout an
 * ensmallen.Graph hands over (.../pecanpy_embedders/node2vec.py:139-163), built without
 * Ensmallen (the reference's only in-tree idiom is the GraphBuilder loop of
 * .../utils/networkx_utils.py:79-113).  indptr receives n_nodes + 1 entries, indices at most
 * indices_capacity entries (2 * n_edges always suffices when symmetrise != 0).
 */
int b2e_csr_from_edges(int device, const uint32_t *src, const uint32_t *dst, uint64_t n_edges,
                       uint64_t n_nodes, int symmetrise, int64_t *indptr, uint32_t *indices,
                       uint64_t indices_capacity, uint64_t *nnz);
/*
 * Same with one float32 weight per input edge (weights == NULL is b2e_csr_from_edges); out_weights
 * receives one per CSR edge, like indices.  The mirror of an edge carries its weight, and a
 * duplicated edge keeps the weight of its first occurrence, taken over the input edges in input
 * order and then their mirrors (embiggen_b200/graph.py: csr_from_edges).  A negative or NaN weight,
 * self-loops included, fails with B2E_ERR_INVALID.
 */
int b2e_csr_from_edges_weighted(int device, const uint32_t *src, const uint32_t *dst, const float *weights,
                                uint64_t n_edges, uint64_t n_nodes, int symmetrise, int64_t *indptr,
                                uint32_t *indices, float *out_weights, uint64_t indices_capacity, uint64_t *nnz);

/*
 * Seeded synthetic graphs of the BASELINE.json shapes: the first n_edges distinct undirected
 * edges, in draw order, of the Philox stream (seed, draw index).  kind 0 = Erdos-Renyi G(n, m);
 * kind 1 = R-MAT over 2^scale ids with ids >= n_nodes rejected, quadrant thresholds
 * t_a = floor(a 2^32), t_ab = floor((a + b) 2^32), t_abc = floor((a + b + c) 2^32).
 * indices_capacity must be at least 2 * n_edges.
 */
int b2e_synthetic_csr(int device, int kind, uint64_t n_nodes, uint32_t scale, uint64_t n_edges,
                      uint64_t seed, uint64_t t_a, uint64_t t_ab, uint64_t t_abc, int64_t *indptr,
                      uint32_t *indices, uint64_t indices_capacity, uint64_t *nnz);

/*
 * Resident graphs: the same builders, but the CSR stays in HBM and is handed to a handle without a
 * copy (SURVEY.md 8(f) row 1: "zero-copy hand-off"; the accessor idiom it replaces is
 * .../pecanpy_embedders/node2vec.py:139-163, which copies both arrays through the host).  A
 * b2e_graph is reference counted: b2e_load_graph makes the handle walk on the graph's own device
 * arrays, b2e_graph_destroy may be called right after it.  b2e_graph_export copies the CSR to host
 * buffers of n + 1 and nnz entries (b2e_graph_shape).
 * A resident graph may carry edge weights (the _weighted builders; never negative): a handle then
 * walks by weight, with its per-row alias tables built on the device from the resident weights.
 * b2e_graph_weighted returns 1 for such a graph, 0 otherwise; b2e_graph_export_weights copies its
 * nnz weights to the host (B2E_ERR_STATE without weights).
 */
typedef struct b2e_graph b2e_graph;
int b2e_graph_from_edges(int device, const uint32_t *src, const uint32_t *dst, uint64_t n_edges,
                         uint64_t n_nodes, int symmetrise, b2e_graph **graph);
int b2e_graph_from_edges_weighted(int device, const uint32_t *src, const uint32_t *dst, const float *weights,
                                  uint64_t n_edges, uint64_t n_nodes, int symmetrise, b2e_graph **graph);
int b2e_graph_synthetic(int device, int kind, uint64_t n_nodes, uint32_t scale, uint64_t n_edges,
                        uint64_t seed, uint64_t t_a, uint64_t t_ab, uint64_t t_abc, b2e_graph **graph);
/* a host CSR uploaded once, e.g. to be shared by the handles of the Walklets scales */
int b2e_graph_from_csr(int device, const int64_t *indptr, const uint32_t *indices, uint64_t n_nodes,
                       uint64_t nnz, b2e_graph **graph);
/* ... with nnz non-negative weights aligned with indices (weights == NULL is b2e_graph_from_csr) */
int b2e_graph_from_csr_weighted(int device, const int64_t *indptr, const uint32_t *indices, const float *weights,
                                uint64_t n_nodes, uint64_t nnz, b2e_graph **graph);
int b2e_graph_shape(const b2e_graph *graph, uint64_t *n_nodes, uint64_t *nnz);
int b2e_graph_export(const b2e_graph *graph, int64_t *indptr, uint32_t *indices);
int b2e_graph_weighted(const b2e_graph *graph);
int b2e_graph_export_weights(const b2e_graph *graph, float *weights);
void b2e_graph_destroy(b2e_graph *graph);
int b2e_load_graph(b2e_handle *handle, b2e_graph *graph);

/* ---- the step after the path: edge embeddings and a perceptron edge scorer (SURVEY.md 8(f) row 4) ---- */

/* EdgeTransformer.methods, .../embedding_transformers/edge_transformer.py:337-350, same order */
typedef enum {
    B2E_EDGE_HADAMARD = 0, B2E_EDGE_SUM = 1, B2E_EDGE_AVERAGE = 2, B2E_EDGE_L1 = 3,
    B2E_EDGE_ABSOLUTE_L1 = 4, B2E_EDGE_SQUARED_L2 = 5, B2E_EDGE_L2 = 6, B2E_EDGE_CONCATENATE = 7,
    B2E_EDGE_MIN = 8, B2E_EDGE_MAX = 9, B2E_EDGE_L2_DISTANCE = 10, B2E_EDGE_COSINE_SIMILARITY = 11
} b2e_edge_method;

/* `edge_features` of PerceptronEdgePrediction (perceptron.py:38-46), computed from the support
 * graph's sorted CSR: Degree = (deg u, deg v) / max degree (two values), Adamic-Adar = sum over
 * the common neighbours of 1 / ln deg, Jaccard = common / union, resource allocation index =
 * sum of 1 / deg, preferential attachment = deg u * deg v / max degree^2.  (Cooccurrence is not
 * implemented.) */
typedef enum {
    B2E_EDGE_FEATURE_DEGREE = 0, B2E_EDGE_FEATURE_ADAMIC_ADAR = 1, B2E_EDGE_FEATURE_JACCARD_COEFFICIENT = 2,
    B2E_EDGE_FEATURE_RESOURCE_ALLOCATION_INDEX = 3, B2E_EDGE_FEATURE_PREFERENTIAL_ATTACHMENT = 4
} b2e_edge_feature;

/* node features (n x dim float32) resident in HBM */
typedef struct b2e_features b2e_features;
int b2e_features_create(int device, const float *host_features, uint64_t n, uint32_t dim,
                        b2e_features **features);
/* zero-copy view of a trained handle's table (0: input table T0, 1: output table T1): the
 * embedding never leaves HBM between b2e_fit and the scorer; valid while the handle lives */
int b2e_features_from_handle(b2e_handle *handle, int table, b2e_features **features);
void b2e_features_destroy(b2e_features *features);

/* width of the concatenation: the methods (Concatenate 2 dim, the two scalar methods 1), then
 * the edge features (Degree 2, the others 1) */
int b2e_edge_embedding_size(uint32_t dim, const uint32_t *methods, uint32_t n_methods,
                            const uint32_t *edge_features, uint32_t n_edge_features, uint32_t *size);

/* the edge features of an edge list, materialised (`graph.get_jaccard_coefficient_scores` and
 * friends, .../visualizations/graph_visualizer.py:2465,2677): out is m x width, host */
int b2e_edge_metrics(int device, const int64_t *indptr, const uint32_t *indices, uint64_t n, uint64_t nnz,
                     const uint32_t *src, const uint32_t *dst, uint64_t m, const uint32_t *edge_features,
                     uint32_t n_edge_features, float *out);

/* EdgeTransformer.transform (edge_transformer.py:352-361): out is m x size, row-major, host */
int b2e_edge_embedding(const b2e_features *features, const uint32_t *src, const uint32_t *dst,
                       uint64_t m, const uint32_t *methods, uint32_t n_methods, float *out);

/* kwargs of PerceptronEdgePrediction that reach the native model
 * (.../edge_prediction/edge_prediction_ensmallen/perceptron.py:18-31, :97-109) */
typedef struct {
    uint32_t struct_size;
    uint32_t n_methods;
    uint32_t methods[12];  /* b2e_edge_method: `edge_embeddings` */
    uint32_t n_edge_features;
    uint32_t edge_features[5]; /* b2e_edge_feature: `edge_features`, appended after the embeddings */
    uint32_t number_of_epochs;
    uint32_t number_of_edges_per_mini_batch;
    float learning_rate;
    float first_order_decay_factor;
    float second_order_decay_factor;
    uint32_t avoid_false_negatives;
    uint32_t use_scale_free_distribution;
} b2e_perceptron_config;

/* `models.EdgePredictionPerceptron(...).fit(graph, node_features)` (perceptron.py:133-170):
 * params receives size weights followed by the bias; epoch_loss (may be NULL) one mean
 * cross-entropy per epoch */
int b2e_perceptron_fit(const b2e_features *features, const int64_t *indptr, const uint32_t *indices,
                       uint64_t n, uint64_t nnz, const b2e_perceptron_config *config, uint64_t seed,
                       float *params, float *epoch_loss);

/* `.predict(graph, node_features)` on an explicit edge list (perceptron.py:172-215); the
 * support graph's CSR is needed only with edge features, the node features only with edge
 * embeddings (either may be NULL otherwise; the same holds for b2e_perceptron_fit's features) */
int b2e_perceptron_predict(const b2e_features *features, const int64_t *indptr, const uint32_t *indices,
                           uint64_t n, uint64_t nnz, const uint32_t *src, const uint32_t *dst, uint64_t m,
                           const uint32_t *methods, uint32_t n_methods, const uint32_t *edge_features,
                           uint32_t n_edge_features, const float *params, float *scores);

#ifdef __cplusplus
}
#endif
#endif
