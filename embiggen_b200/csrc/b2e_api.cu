// C ABI of the engine (include/b2e.h): handle management, K1 CSR upload, K3 alias table,
// the chunked walk -> SGD pipeline on two streams, and the host-buffer entry points.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <functional>
#include <new>

#include "host.cuh"

using namespace b2e;

#define REQUIRE_HANDLE(h)                                                                    \
    do {                                                                                     \
        if (!(h)) return fail(B2E_ERR_INVALID, "null handle");                               \
        CUDA_TRY(cudaSetDevice((h)->cfg.device));                                            \
    } while (0)

extern "C" const char *b2e_last_error(void) { return g_last_error.c_str(); }
extern "C" int b2e_abi_version(void) { return B2E_ABI_VERSION; }

extern "C" int b2e_device_count(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) return 0;
    int usable = 0;
    for (int d = 0; d < count; ++d) {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, d) == cudaSuccess && prop.major >= 10) ++usable;
    }
    return usable;
}

extern "C" int b2e_select_device(int device) { return select_device(device); }

// an accept probability r as an integer threshold: floor(r 2^32), clamped to 2^32
static unsigned long long quantise(double r) {
    const double t = floor(r * 4294967296.0);
    return t >= 4294967296.0 ? 4294967296ull : (unsigned long long)t;
}

// accept thresholds of the typed-walk tests, [same type, changed type] (oracle/walks.c)
static void type_thresholds(float change_weight, unsigned long long q[2]) {
    const double w = (double)change_weight, m = w > 1.0 ? w : 1.0;
    q[0] = quantise(1.0 / m);
    q[1] = quantise(w / m);
}

static bool walklet(const b2e_config &c) { return c.walklet_scale >= 2; }
static uint32_t sub_walk_length(const b2e_config &c) {
    return walklet(c) ? (c.walk_length + c.walklet_scale - 1) / c.walklet_scale : c.walk_length;
}

// integer accept thresholds (DESIGN.md "second-order accept test")
static void thresholds(float return_weight, float explore_weight, unsigned long long out[3]) {
    const double w[3] = {(double)return_weight, 1.0, (double)explore_weight};
    const double wmax = std::max(w[0], std::max(w[1], w[2]));
    for (int i = 0; i < 3; ++i) out[i] = quantise(w[i] / wmax);  // w[i] = wmax gives exactly 2^32
}

// folded return edge (oracle/walks.c: orc_fold_thresholds): accept thresholds against the envelope
// of the non-return classes, and the excess E of the return edge in units of 2^-20 envelopes
static void fold_thresholds(float return_weight, float explore_weight, unsigned long long out[3],
                            uint64_t *excess) {
    const double rw = (double)return_weight, ew = (double)explore_weight;
    const double wenv = ew > 1.0 ? ew : 1.0;
    const double w[3] = {wenv, 1.0, ew};
    for (int i = 0; i < 3; ++i) out[i] = quantise(w[i] / wenv);
    double e = rw > wenv ? floor((rw - wenv) / wenv * 1048576.0) : 0.0;
    if (e > 2147483648.0) e = 2147483648.0;
    *excess = (uint64_t)e;
}

extern "C" int b2e_create(const b2e_config *config, b2e_handle **out) {
    if (!config || !out) return fail(B2E_ERR_INVALID, "null argument");
    if (config->struct_size != sizeof(b2e_config))
        return fail(B2E_ERR_INVALID, "b2e_config.struct_size does not match this library (ABI mismatch)");
    const b2e_config &c = *config;
    if (c.model > B2E_GLOVE) return fail(B2E_ERR_INVALID, "model must be 0 (SkipGram), 1 (CBOW) or 2 (GloVe)");
    if (c.model == B2E_GLOVE && (c.walklet_scale >= 2 || c.stochastic_downsample_by_degree))
        return fail(B2E_ERR_INVALID, "GloVe supports neither walklet_scale nor stochastic_downsample_by_degree");
    if (c.model == B2E_GLOVE && !(c.glove_alpha >= 0.0f))
        return fail(B2E_ERR_INVALID, "glove_alpha must be non-negative");
    if (c.embedding_size == 0 || c.embedding_size > 512)
        return fail(B2E_ERR_INVALID, "embedding_size must be in [1, 512]");
    if (c.walk_length < 2 || c.walk_length > 65535)
        return fail(B2E_ERR_INVALID, "walk_length must be in [2, 65535]");
    if (c.walklet_scale >= c.walk_length)
        return fail(B2E_ERR_INVALID, "walklet_scale must be smaller than walk_length");
    if (c.window_size == 0 || c.window_size > 64)
        return fail(B2E_ERR_INVALID, "window_size must be in [1, 64]");
    if (c.number_of_negative_samples > 31)
        return fail(B2E_ERR_INVALID, "number_of_negative_samples must be at most 31");
    if (c.shared_negatives) {
        if (c.model != B2E_SKIPGRAM)
            return fail(B2E_ERR_INVALID, "shared_negatives is a SkipGram option (CBOW already draws per centre)");
        if (c.window_size > 7 || c.number_of_negative_samples > 15 || c.embedding_size > 128 ||
            sub_walk_length(c) > 1024)
            return fail(B2E_ERR_INVALID, "shared_negatives needs window_size <= 7, number_of_negative_samples <= 15, "
                                         "embedding_size <= 128 and walk_length <= 1024");
    }
    if (c.iterations == 0) return fail(B2E_ERR_INVALID, "iterations must be positive");
    if (!(c.return_weight > 0.0f) || !(c.explore_weight > 0.0f))
        return fail(B2E_ERR_INVALID, "return_weight and explore_weight must be strictly positive");
    if (!(c.change_node_type_weight > 0.0f) || !(c.change_edge_type_weight > 0.0f))
        return fail(B2E_ERR_INVALID, "change_node_type_weight and change_edge_type_weight must be strictly positive");
    if (!(c.clipping_value > 0.0f)) return fail(B2E_ERR_INVALID, "clipping_value must be positive");
    if (!(c.negative_sampling_exponent >= 0.0f))
        return fail(B2E_ERR_INVALID, "negative_sampling_exponent must be non-negative");

    if (int rc = select_device(c.device)) return rc;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, c.device));
    if (prop.major < 10)
        return fail(B2E_ERR_CUDA, "this library is built for sm_100a (Blackwell) only");

    b2e_handle *h = new (std::nothrow) b2e_handle();
    if (!h) return fail(B2E_ERR_INVALID, "out of host memory");
    h->cfg = c;
    h->sm_count = prop.multiProcessorCount;
    // rows start on 128 B lines: a random row then touches the fewest lines (measured with
    // scripts/microbench_rows: +13 % rows/s over a dense 400 B pitch for D = 100)
    h->row_stride = (c.embedding_size + 31u) / 32u * 32u;
    thresholds(c.return_weight, c.explore_weight, h->thr);
    h->second_order = !(c.return_weight == 1.0f && c.explore_weight == 1.0f);
    for (int s = 0; s < 2; ++s) {
        if (cudaEventCreateWithFlags(&h->walk_done[s], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&h->train_done[s], cudaEventDisableTiming) != cudaSuccess) {
            b2e_destroy(h);
            return fail(B2E_ERR_CUDA, "cudaEventCreate failed");
        }
    }
    if (cudaStreamCreateWithFlags(&h->walk_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->train_stream, cudaStreamNonBlocking) != cudaSuccess ||
        h->d_counters.reserve(sizeof(DeviceCounters)) != cudaSuccess ||
        cudaMemsetAsync(h->d_counters.get(), 0, sizeof(DeviceCounters), h->train_stream) != cudaSuccess ||
        cudaStreamSynchronize(h->train_stream) != cudaSuccess) {
        b2e_destroy(h);
        return fail(B2E_ERR_CUDA, "stream / counter allocation failed");
    }
    h->own_streams = true;
    *out = h;
    return B2E_OK;
}

static void close_peers(b2e_handle *h) {
    for (uint32_t g = 0; g < B2E_MAX_WORLD; ++g) {
        if (h->peers_are_ipc && g != h->rank) {
            if (h->peer_t0[g]) cudaIpcCloseMemHandle(h->peer_t0[g]);
            if (h->peer_t1[g]) cudaIpcCloseMemHandle(h->peer_t1[g]);
        }
        h->peer_t0[g] = h->peer_t1[g] = nullptr;
    }
    h->world = 1;
    h->rank = 0;
    h->peers_are_ipc = false;
}

static int require_graph(b2e_handle *h) {
    if (!h->graph.csr) return fail(B2E_ERR_STATE, "b2e_load_csr must be called first");
    return B2E_OK;
}

static void drop_graph(b2e_handle *h) {
    close_peers(h);
    h->graph = HandleGraph();
}

extern "C" void b2e_destroy(b2e_handle *h) {
    if (!h) return;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    drop_graph(h);
    for (int s = 0; s < 2; ++s) {
        if (h->walk_done[s]) cudaEventDestroy(h->walk_done[s]);
        if (h->train_done[s]) cudaEventDestroy(h->train_done[s]);
    }
    if (h->own_streams) {
        if (h->walk_stream) cudaStreamDestroy(h->walk_stream);
        if (h->train_stream) cudaStreamDestroy(h->train_stream);
    }
    delete h;
}

extern "C" int b2e_load_types(b2e_handle *h, const uint32_t *node_types, const uint32_t *edge_types) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    h->graph.node_types.reset();
    h->graph.edge_types.reset();
    if (node_types && h->n) {
        CUDA_TRY(h->graph.node_types.reserve(h->n * sizeof(uint32_t)));
        CUDA_TRY(cudaMemcpyAsync(h->graph.node_types.get(), node_types, h->n * sizeof(uint32_t),
                                 cudaMemcpyHostToDevice, h->walk_stream));
    }
    if (edge_types && h->nnz) {
        CUDA_TRY(h->graph.edge_types.reserve(h->nnz * sizeof(uint32_t)));
        CUDA_TRY(cudaMemcpyAsync(h->graph.edge_types.get(), edge_types, h->nnz * sizeof(uint32_t),
                                 cudaMemcpyHostToDevice, h->walk_stream));
    }
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));  // the caller's buffers may go away
    return B2E_OK;
}

extern "C" int b2e_load_csr(b2e_handle *h, const int64_t *indptr, const uint32_t *indices,
                            uint64_t n, uint64_t nnz) {
    return b2e_load_csr_weighted(h, indptr, indices, nullptr, n, nnz);
}

// Everything a load builds on the device once the old graph is gone.  `d_flags` belongs to the
// caller, so that a failed load frees it only after the device has been drained.
static int build_graph(b2e_handle *h, const int64_t *indptr, const uint32_t *indices, const float *weights,
                       b2e_graph *resident, DeviceBuffer<int> &d_flags,
                       const std::function<void(const char *)> &lap) {
    const b2e_config &c = h->cfg;
    const uint64_t n = h->n, nnz = h->nnz;
    HandleGraph &g = h->graph;
    // K1: the two big copies into a graph of this handle's own (none when the CSR is resident
    // already), then the checks on the device: offsets non-decreasing and within nnz; ids in
    // range, rows strictly ascending (the kernels index with these ids and bisect these rows
    // without looking again)
    if (resident) {
        ++resident->references;
        g.csr.reset(resident);
    } else {
        g.csr.reset(new b2e_graph());
        ResidentCsr &upload = g.csr->csr;
        g.csr->device = c.device;
        upload.n = n;
        upload.nnz = nnz;
        CUDA_TRY(upload.indptr.reserve((n + 1) * sizeof(int64_t)));
        CUDA_TRY(upload.indices.reserve(nnz * sizeof(uint32_t)));
        CUDA_TRY(cudaMemcpyAsync(upload.indptr.get(), indptr, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice,
                                 h->walk_stream));
        CUDA_TRY(cudaMemcpyAsync(upload.indices.get(), indices, nnz * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                 h->walk_stream));
    }
    const int64_t *d_indptr = g.csr->csr.indptr.get();
    const uint32_t *d_indices = g.csr->csr.indices.get();
    int flags[2] = {0, 1};
    CUDA_TRY(d_flags.reserve(2 * sizeof(int)));
    CUDA_TRY(cudaMemsetAsync(d_flags.get(), 0, 2 * sizeof(int), h->walk_stream));
    CUDA_TRY(check_indptr_device(d_indptr, n, nnz, d_flags.get(), h->walk_stream));
    CUDA_TRY(cudaMemcpyAsync(flags, d_flags.get(), sizeof(int), cudaMemcpyDeviceToHost, h->walk_stream));
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    if (flags[0]) return fail(B2E_ERR_INVALID, "indptr must be non-decreasing and end at nnz");
    CUDA_TRY(launch_csr_check(d_indptr, d_indices, n, d_flags.get(), h->sm_count, h->walk_stream));
    h->launches += 2;
    CUDA_TRY(cudaMemcpyAsync(flags, d_flags.get(), sizeof(int), cudaMemcpyDeviceToHost, h->walk_stream));
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    lap("CSR upload + content checks");
    if (flags[0]) {
        return fail(B2E_ERR_INVALID, flags[0] & 1 ? "a destination node id is out of range"
                                                  : "neighbour lists must be sorted strictly ascending within each row");
    }

    // K3 on the device: start nodes, maximum degree, alias table over deg^alpha (alias_build.cu)
    h->h_alias_thr.clear();
    h->h_alias_idx.clear();
    {
        DeviceBuffer<uint32_t> sources_all;
        CUDA_TRY(sources_all.reserve(n * sizeof(uint32_t)));
        if (c.use_scale_free_distribution && g.alias.reserve(n * sizeof(uint2)) != cudaSuccess)
            return fail(B2E_ERR_CUDA, "out of device memory (alias table)");
        std::string error;
        uint64_t n_src = 0, max_degree = 0;
        const cudaError_t e = build_node_tables(d_indptr, indptr, n, (double)c.negative_sampling_exponent,
                                                sources_all.get(), &n_src, &max_degree, g.alias.get(), h->walk_stream,
                                                error);
        if (e != cudaSuccess) return fail(e == cudaErrorInvalidValue ? B2E_ERR_INVALID : B2E_ERR_CUDA, error);
        CUDA_TRY(g.sources.reserve(std::max<uint64_t>(1, n_src) * sizeof(uint32_t)));
        if (n_src)
            CUDA_TRY(cudaMemcpy(g.sources.get(), sources_all.get(), n_src * sizeof(uint32_t), cudaMemcpyDeviceToDevice));
        h->n_src = n_src;
        h->max_degree = (uint32_t)std::min<uint64_t>(max_degree, 0xFFFFFFFEull);
        h->launches += 8;
    }
    lap("start nodes + alias table (GPU)");

    // Edge weights: the per-row alias tables of the proposal, built on the device (alias_build.cu)
    // from the resident graph's own weights or from host weights uploaded once (4 B per edge,
    // freed once the table is built).  normalize_by_degree (.../node2vec_skipgram.py:94-96) divides the
    // weight of v -> x by max(deg(x), 1), one float32 division per edge on the device, folded into
    // the proposal table -- no extra rejection however skewed the degrees (oracle:
    // degree_normalised_weights).
    const float *d_weights = g.csr->csr.weights.get();
    DeviceBuffer<float> uploaded, normalised;
    if (weights) {
        CUDA_TRY(uploaded.reserve(nnz * sizeof(float)));
        CUDA_TRY(cudaMemcpyAsync(uploaded.get(), weights, nnz * sizeof(float), cudaMemcpyHostToDevice, h->walk_stream));
        d_weights = uploaded.get();
        lap("edge weight upload");
    }
    if (c.normalize_by_degree) {
        CUDA_TRY(normalised.reserve(nnz * sizeof(float)));
        CUDA_TRY(launch_degree_normalise(d_indptr, d_indices, d_weights, nnz, normalised.get(), h->walk_stream));
        ++h->launches;
        d_weights = normalised.get();
        lap("degree normalisation (GPU)");
    }
    if (d_weights) {
        CUDA_TRY(g.edge_alias.reserve(nnz * sizeof(uint2)));
        std::string error;
        uint64_t longest_row = 0;
        const cudaError_t e = build_edge_alias(d_indptr, d_weights, n, nnz, g.edge_alias.get(), &longest_row,
                                               h->walk_stream, error);
        if (e != cudaSuccess) return fail(e == cudaErrorInvalidValue ? B2E_ERR_INVALID : B2E_ERR_CUDA, error);
        h->launches += 3;
        lap(("edge alias tables (GPU, longest row " + std::to_string(longest_row) + ")").c_str());
    }
    const bool weighted = d_weights != nullptr;
    uploaded.reset();  // the table is built: a host load's weights and the normalised ones go
    normalised.reset();
    // Second-order walks: is the graph undirected (every edge mirrored)?  Verified here, never
    // assumed: it allows the adjacency check in the shorter of the two rows and the folded return
    // edge.  The row filters answer most adjacency checks with one gather (walk_kernels.cu).
    h->undirected = false;
    h->fold_excess = 0;
    if (h->second_order) {
        if (!getenv("B2E_ASSUME_DIRECTED")) {
            CUDA_TRY(cudaMemcpyAsync(d_flags.get() + 1, flags + 1, sizeof(int), cudaMemcpyHostToDevice, h->walk_stream));
            CUDA_TRY(launch_symmetry_check(d_indptr, d_indices, n, nnz, d_flags.get() + 1, h->walk_stream));
            CUDA_TRY(cudaMemcpyAsync(flags + 1, d_flags.get() + 1, sizeof(int), cudaMemcpyDeviceToHost, h->walk_stream));
            CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
            h->undirected = flags[1] != 0;
            ++h->launches;
            lap("symmetry check");
        }
        uint64_t excess = 0;
        fold_thresholds(c.return_weight, c.explore_weight, h->thr_fold, &excess);
        if (h->undirected && !weighted && !getenv("B2E_NO_FOLD")) h->fold_excess = excess;
        if (!getenv("B2E_NO_FILTER")) {
            const uint64_t words = row_filter_words(nnz);
            CUDA_TRY(g.filter.reserve(words * sizeof(unsigned long long)));
            CUDA_TRY(cudaMemsetAsync(g.filter.get(), 0, words * sizeof(unsigned long long), h->walk_stream));
            CUDA_TRY(launch_row_filter_build(d_indptr, d_indices, n, g.filter.get(), h->sm_count, h->walk_stream));
            ++h->launches;
        }
    }
    lap("row filters");

    CUDA_TRY(g.t0.reserve(n * (uint64_t)h->row_stride * sizeof(float)));
    CUDA_TRY(g.t1.reserve(n * (uint64_t)h->row_stride * sizeof(float)));

    const uint64_t per_epoch = (uint64_t)c.iterations * h->n_src;
    // an explicit chunk_walks is honoured as given (parity tests feed host walks of that size)
    const uint64_t cap = c.chunk_walks ? c.chunk_walks
                                       : std::max<uint64_t>(1, std::min<uint64_t>(1ull << 20, per_epoch));
    h->chunk_cap = cap;
    // Walklets: a slot holds the k sub-walks of every walk, k * ceil(L / k) >= L tokens per walk
    const uint64_t slot_tokens = walklet(c) ? (uint64_t)c.walklet_scale * sub_walk_length(c) : c.walk_length;
    for (int s = 0; s < 2; ++s)
        CUDA_TRY(g.walks[s].reserve(cap * slot_tokens * sizeof(uint32_t)));
    if (walklet(c)) CUDA_TRY(g.walk_raw.reserve(cap * c.walk_length * sizeof(uint32_t)));
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    lap("tables + walk ring allocation");
    return B2E_OK;
}

// `resident`: the CSR already lives in HBM (b2e_load_graph) -- `indptr` is a host copy of its
// offsets, `indices` is null and nothing is uploaded
static int load_graph_common(b2e_handle *h, const int64_t *indptr, const uint32_t *indices, const float *weights,
                             uint64_t n, uint64_t nnz, b2e_graph *resident) {
    if (n == 0) return fail(B2E_ERR_INVALID, "The provided graph is empty.");
    if (n >= 0xFFFFFF00ull) return fail(B2E_ERR_INVALID, "node ids must be below 0xFFFFFF00");
    if (nnz == 0) return fail(B2E_ERR_INVALID, "The provided graph does not have edges.");
    if (indptr && (indptr[0] != 0 || (uint64_t)indptr[n] != nnz))
        return fail(B2E_ERR_INVALID, "indptr must start at 0 and end at nnz");
    // B2E_LOAD_TIMING=1: where the time of a load goes, on stderr
    const bool timing = getenv("B2E_LOAD_TIMING") != nullptr;
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double mark = now();
    auto lap = [&](const char *what) {
        if (!timing) return;
        cudaDeviceSynchronize();
        const double t = now();
        fprintf(stderr, "[b2e load] %-28s %8.3f s\n", what, t - mark);
        mark = t;
    };
    if (weights)
        for (uint64_t e = 0; e < nnz; ++e)
            if (!(weights[e] >= 0.0f)) return fail(B2E_ERR_INVALID, "edge weights must be non-negative numbers");

    CUDA_TRY(cudaDeviceSynchronize());
    drop_graph(h);
    h->n = n;
    h->nnz = nnz;
    DeviceBuffer<int> d_flags;
    const int rc = build_graph(h, indptr, indices, weights, resident, d_flags, lap);
    if (rc != B2E_OK) {  // a failed load leaves the handle without a graph (require_graph() then fails cleanly)
        cudaDeviceSynchronize();
        drop_graph(h);
        h->n = h->nnz = h->n_src = 0;
    }
    return rc;
}

extern "C" int b2e_load_csr_weighted(b2e_handle *h, const int64_t *indptr, const uint32_t *indices,
                                     const float *weights, uint64_t n, uint64_t nnz) {
    REQUIRE_HANDLE(h);
    if (!indptr || (!indices && nnz)) return fail(B2E_ERR_INVALID, "null CSR pointer");
    return load_graph_common(h, indptr, indices, weights, n, nnz, nullptr);
}

extern "C" uint64_t b2e_number_of_sources(const b2e_handle *h) { return h ? h->n_src : 0; }
extern "C" uint64_t b2e_row_stride(const b2e_handle *h) { return h ? h->row_stride : 0; }
extern "C" uint64_t b2e_launch_count(const b2e_handle *h) { return h ? h->launches : 0; }

extern "C" int b2e_chunk_capacity(const b2e_handle *h, uint64_t *walks) {
    if (!h || !walks) return fail(B2E_ERR_INVALID, "null argument");
    *walks = h->chunk_cap;
    return B2E_OK;
}

extern "C" int b2e_set_streams(b2e_handle *h, void *walk_stream, void *train_stream) {
    REQUIRE_HANDLE(h);
    CUDA_TRY(cudaDeviceSynchronize());
    if (h->own_streams) {
        cudaStreamDestroy(h->walk_stream);
        cudaStreamDestroy(h->train_stream);
        h->own_streams = false;
    }
    h->walk_stream = (cudaStream_t)walk_stream;
    h->train_stream = (cudaStream_t)train_stream;
    return B2E_OK;
}

extern "C" int b2e_init_tables(b2e_handle *h, uint64_t seed) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    CUDA_TRY(launch_init_tables(h->graph.t0.get(), h->graph.t1.get(), h->n, h->cfg.embedding_size, h->row_stride, seed,
                                h->train_stream));
    ++h->launches;
    return B2E_OK;
}

static int walk_into(b2e_handle *h, uint64_t seed, uint64_t first_walk, uint64_t n_walks,
                     uint64_t walk_id_stride, uint32_t *d_out, cudaStream_t stream) {
    WalkParams p;
    p.indptr = h->graph.csr->csr.indptr.get();
    p.indices = h->graph.csr->csr.indices.get();
    p.edge_alias = h->graph.edge_alias.get();
    p.node_types = h->graph.node_types.get();
    p.edge_types = h->graph.edge_types.get();
    type_thresholds(h->graph.node_types.get() ? h->cfg.change_node_type_weight : 1.0f, p.q_node);
    type_thresholds(h->graph.edge_types.get() ? h->cfg.change_edge_type_weight : 1.0f, p.q_edge);
    p.sources = h->graph.sources.get();
    p.n_src = h->n_src;
    p.seed_lo = (uint32_t)seed;
    p.seed_hi = (uint32_t)(seed >> 32);
    p.first_walk = first_walk;
    p.n_walks = n_walks;
    p.walk_id_stride = walk_id_stride;
    p.walk_length = h->cfg.walk_length;
    // typed walks keep the plain envelope (their trial loop has its own Philox layout)
    const bool typed = (h->graph.node_types.get() && p.q_node[0] != p.q_node[1]) || (h->graph.edge_types.get() && p.q_edge[0] != p.q_edge[1]);
    const unsigned long long *thr = h->fold_excess && !typed ? h->thr_fold : h->thr;
    p.fold_excess = typed ? 0 : h->fold_excess;
    p.filter = h->graph.filter.get();
    p.thr_return = thr[0];
    p.thr_common = thr[1];
    p.thr_explore = thr[2];
    p.out = d_out;
    p.counters = h->d_counters.get();
    p.undirected = h->undirected ? 1u : 0u;
    p.sm_count = h->sm_count;
    CUDA_TRY(launch_walks(p, h->second_order, stream));
    if (n_walks) ++h->launches;
    return B2E_OK;
}

extern "C" int b2e_walk_chunk(b2e_handle *h, uint64_t seed, uint64_t first_walk, uint64_t n_walks,
                              uint64_t walk_id_stride, uint32_t slot) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (slot > 1) return fail(B2E_ERR_INVALID, "slot must be 0 or 1");
    if (n_walks > h->chunk_cap) return fail(B2E_ERR_INVALID, "n_walks exceeds the chunk capacity");
    if (walk_id_stride == 0) return fail(B2E_ERR_INVALID, "walk_id_stride must be positive");
    if (h->n_src == 0) return fail(B2E_ERR_INVALID, "the graph has no node with outgoing edges");
    // the slot may still be read by the SGD kernel of two chunks ago
    CUDA_TRY(cudaStreamWaitEvent(h->walk_stream, h->train_done[slot], 0));
    uint32_t *target = walklet(h->cfg) ? h->graph.walk_raw.get() : h->graph.walks[slot].get();
    if (int rc = walk_into(h, seed, first_walk, n_walks, walk_id_stride, target, h->walk_stream))
        return rc;
    if (walklet(h->cfg)) {
        CUDA_TRY(launch_walklet_split(h->graph.walk_raw.get(), n_walks, h->cfg.walk_length, h->cfg.walklet_scale,
                                      h->graph.walks[slot].get(), h->walk_stream));
        if (n_walks) ++h->launches;
    }
    CUDA_TRY(cudaEventRecord(h->walk_done[slot], h->walk_stream));
    h->slot_first[slot] = first_walk;
    h->slot_count[slot] = n_walks;
    h->slot_stride[slot] = walk_id_stride;
    return B2E_OK;
}

// Walklets in one pass: every scale has its own handle (its own tables), but the walks of a chunk
// are the same for all of them -- `dst` takes the chunk `src` has just walked into `slot` instead
// of walking it again (split by its own scale, or copied), ordered after src's walk on the device.
extern "C" int b2e_adopt_walks(b2e_handle *dst, b2e_handle *src, uint32_t slot) {
    REQUIRE_HANDLE(dst);
    if (!src) return fail(B2E_ERR_INVALID, "null source handle");
    if (int rc = require_graph(dst)) return rc;
    if (int rc = require_graph(src)) return rc;
    if (slot > 1) return fail(B2E_ERR_INVALID, "slot must be 0 or 1");
    if (src->cfg.device != dst->cfg.device || src->cfg.walk_length != dst->cfg.walk_length)
        return fail(B2E_ERR_INVALID, "both handles must sit on one device and use one walk_length");
    const uint64_t n_walks = src->slot_count[slot];
    if (n_walks > dst->chunk_cap) return fail(B2E_ERR_INVALID, "the chunk exceeds the capacity of the adopting handle");
    const uint32_t L = dst->cfg.walk_length;
    const uint32_t *raw = walklet(src->cfg) ? src->graph.walk_raw.get() : src->graph.walks[slot].get();
    CUDA_TRY(cudaStreamWaitEvent(dst->walk_stream, src->walk_done[slot], 0));
    CUDA_TRY(cudaStreamWaitEvent(dst->walk_stream, dst->train_done[slot], 0));
    if (walklet(dst->cfg)) {
        CUDA_TRY(launch_walklet_split(raw, n_walks, L, dst->cfg.walklet_scale, dst->graph.walks[slot].get(), dst->walk_stream));
        if (n_walks) ++dst->launches;
    } else {
        CUDA_TRY(cudaMemcpyAsync(dst->graph.walks[slot].get(), raw, n_walks * L * sizeof(uint32_t), cudaMemcpyDeviceToDevice,
                                 dst->walk_stream));
    }
    CUDA_TRY(cudaEventRecord(dst->walk_done[slot], dst->walk_stream));
    dst->slot_first[slot] = src->slot_first[slot];
    dst->slot_count[slot] = n_walks;
    dst->slot_stride[slot] = src->slot_stride[slot];
    return B2E_OK;
}

static int train_slot(b2e_handle *h, uint64_t seed, uint32_t slot, float learning_rate) {
    const b2e_config &c = h->cfg;
    if (c.model == B2E_GLOVE)
        return fail(B2E_ERR_STATE, "a GloVe handle trains with b2e_cooccurrence + b2e_glove_train");
    TrainParams p;
    p.walks = h->graph.walks[slot].get();
    p.first_walk = h->slot_first[slot];
    p.n_walks = h->slot_count[slot];
    p.walk_id_stride = h->slot_stride[slot];
    p.seed_lo = (uint32_t)seed;
    p.seed_hi = (uint32_t)(seed >> 32);
    p.n = (uint32_t)h->n;
    p.walk_length = sub_walk_length(c);
    p.window = c.window_size;
    p.negatives = c.number_of_negative_samples;
    p.row_stride = h->row_stride;
    p.chunks = (c.embedding_size + 3u) / 4u;
    p.clip = c.clipping_value;
    p.lr = learning_rate;
    p.inv_scale = 1.0f / sqrtf((float)c.embedding_size);
    p.use_alias = c.use_scale_free_distribution ? 1u : 0u;
    p.normalize_lr = c.normalize_learning_rate_by_degree ? 1u : 0u;
    p.downsample = c.stochastic_downsample_by_degree ? h->max_degree + 1u : 0u;
    p.scale_dot = c.scale_by_sqrt_dim ? 1u : 0u;
    p.shared_negatives = c.shared_negatives ? 1u : 0u;
    p.alias = h->graph.alias.get();
    p.indptr = h->graph.csr->csr.indptr.get();
    p.t0 = h->graph.t0.get();
    p.t1 = h->graph.t1.get();
    p.counters = h->d_counters.get();
    // Hogwild staleness: on a tiny graph thousands of concurrent walks would all train against
    // nearly the same stale rows, which slows the first epochs down (the final quality is not
    // affected: scripts/exp_concurrency.py).  Unless told otherwise keep about one walk in flight
    // per 16 nodes for SkipGram and per 64 nodes for CBOW, whose averaged context rows make it
    // lag more; graphs above ~50 k (200 k) nodes are not limited: < 3 000 warps are resident.
    const uint64_t per_walk_nodes = c.model == B2E_CBOW ? 64 : 16;
    const uint64_t max_warps = c.max_concurrent_walks ? c.max_concurrent_walks
                                                       : std::max<uint64_t>(16, h->n / per_walk_nodes);
    // Walklets: one launch per residue r; sub-walk r of walk g draws its negatives as walk
    // g + r * 2^48 (walk ids stay far below 2^48), the slot is laid out [r][walk][token]
    const uint32_t passes = walklet(c) ? c.walklet_scale : 1u;
    for (uint32_t r = 0; r < passes; ++r) {
        p.walks = h->graph.walks[slot].get() + (uint64_t)r * p.n_walks * p.walk_length;
        p.first_walk = h->slot_first[slot] + ((uint64_t)r << 48);
        CUDA_TRY(launch_train(p, c.model, c.deterministic != 0, h->sm_count, max_warps, h->train_stream));
        if (p.n_walks) ++h->launches;
    }
    return B2E_OK;
}

extern "C" int b2e_train_chunk(b2e_handle *h, uint64_t seed, uint32_t slot, float learning_rate) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (slot > 1) return fail(B2E_ERR_INVALID, "slot must be 0 or 1");
    CUDA_TRY(cudaStreamWaitEvent(h->train_stream, h->walk_done[slot], 0));
    if (int rc = train_slot(h, seed, slot, learning_rate)) return rc;
    CUDA_TRY(cudaEventRecord(h->train_done[slot], h->train_stream));
    return B2E_OK;
}

extern "C" int b2e_train_host_walks(b2e_handle *h, uint64_t seed, const uint32_t *walks,
                                    uint64_t first_walk, uint64_t n_walks, uint64_t walk_id_stride,
                                    float learning_rate) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (!walks) return fail(B2E_ERR_INVALID, "null walks");
    if (n_walks > h->chunk_cap) return fail(B2E_ERR_INVALID, "n_walks exceeds the chunk capacity");
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    uint32_t *target = walklet(h->cfg) ? h->graph.walk_raw.get() : h->graph.walks[0].get();
    CUDA_TRY(cudaMemcpyAsync(target, walks, n_walks * h->cfg.walk_length * sizeof(uint32_t),
                             cudaMemcpyHostToDevice, h->train_stream));  // ordered before the kernel
    if (walklet(h->cfg))
        CUDA_TRY(launch_walklet_split(h->graph.walk_raw.get(), n_walks, h->cfg.walk_length, h->cfg.walklet_scale,
                                      h->graph.walks[0].get(), h->train_stream));
    h->slot_first[0] = first_walk;
    h->slot_count[0] = n_walks;
    h->slot_stride[0] = walk_id_stride;
    if (int rc = train_slot(h, seed, 0, learning_rate)) return rc;
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    return B2E_OK;
}

extern "C" int b2e_slot_walks(b2e_handle *h, uint32_t slot, uint64_t n_walks, uint32_t *out) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (slot > 1) return fail(B2E_ERR_INVALID, "slot must be 0 or 1");
    if (walklet(h->cfg)) return fail(B2E_ERR_INVALID, "Walklets slots hold split walks");
    if (!out && n_walks) return fail(B2E_ERR_INVALID, "null output buffer");
    if (n_walks > h->slot_count[slot]) return fail(B2E_ERR_INVALID, "n_walks exceeds the walks in the slot");
    if (int rc = b2e_sync(h)) return rc;
    CUDA_TRY(cudaMemcpyAsync(out, h->graph.walks[slot].get(), n_walks * h->cfg.walk_length * sizeof(uint32_t),
                             cudaMemcpyDeviceToHost, h->train_stream));
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    return B2E_OK;
}

extern "C" int b2e_sync(b2e_handle *h) {
    REQUIRE_HANDLE(h);
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    return B2E_OK;
}

extern "C" int b2e_walks(b2e_handle *h, uint64_t seed, uint64_t first_walk, uint64_t n_walks,
                         uint64_t walk_id_stride, uint32_t *out) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (!out && n_walks) return fail(B2E_ERR_INVALID, "null output buffer");
    if (walk_id_stride == 0) return fail(B2E_ERR_INVALID, "walk_id_stride must be positive");
    if (h->n_src == 0) return fail(B2E_ERR_INVALID, "the graph has no node with outgoing edges");
    if (int rc = b2e_sync(h)) return rc;
    const uint32_t L = h->cfg.walk_length;
    uint64_t done = 0;
    while (done < n_walks) {
        const uint64_t count = std::min(h->chunk_cap, n_walks - done);
        if (int rc = walk_into(h, seed, first_walk + done * walk_id_stride, count, walk_id_stride,
                               h->graph.walks[0].get(), h->walk_stream))
            return rc;
        CUDA_TRY(cudaMemcpyAsync(out + done * L, h->graph.walks[0].get(), count * L * sizeof(uint32_t),
                                 cudaMemcpyDeviceToHost, h->walk_stream));
        CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
        done += count;
    }
    return B2E_OK;
}

extern "C" int b2e_device_tables(b2e_handle *h, void **table0, void **table1) {
    if (!h || !table0 || !table1) return fail(B2E_ERR_INVALID, "null argument");
    if (int rc = require_graph(h)) return rc;
    *table0 = h->graph.t0.get();
    *table1 = h->graph.t1.get();
    return B2E_OK;
}

extern "C" int b2e_host_register(void *buffer, uint64_t bytes) {
    if (!buffer || !bytes) return fail(B2E_ERR_INVALID, "null or empty buffer");
    CUDA_TRY(cudaHostRegister(buffer, bytes, cudaHostRegisterPortable));
    return B2E_OK;
}

extern "C" int b2e_host_unregister(void *buffer) {
    if (!buffer) return fail(B2E_ERR_INVALID, "null buffer");
    CUDA_TRY(cudaHostUnregister(buffer));
    return B2E_OK;
}

// ---- the exchange step (csrc/exchange.cu) ----
extern "C" int b2e_exchange_handles(b2e_handle *h, void *ipc_handles) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (!ipc_handles) return fail(B2E_ERR_INVALID, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == B2E_IPC_HANDLE_BYTES, "B2E_IPC_HANDLE_BYTES");
    cudaIpcMemHandle_t *out = static_cast<cudaIpcMemHandle_t *>(ipc_handles);
    CUDA_TRY(cudaIpcGetMemHandle(out, h->graph.t0.get()));
    CUDA_TRY(cudaIpcGetMemHandle(out + 1, h->graph.t1.get()));
    return B2E_OK;
}

static int check_world(uint32_t world, uint32_t rank) {
    if (world < 1 || world > B2E_MAX_WORLD) return fail(B2E_ERR_INVALID, "world must be in [1, B2E_MAX_WORLD]");
    if (rank >= world) return fail(B2E_ERR_INVALID, "rank must be below world");
    return B2E_OK;
}

extern "C" int b2e_exchange_open(b2e_handle *h, uint32_t world, uint32_t rank, const void *all_ipc_handles) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (int rc = check_world(world, rank)) return rc;
    if (!all_ipc_handles) return fail(B2E_ERR_INVALID, "null argument");
    // nothing mapped yet: no need to drain the device (the caller may have SGD chunks queued and
    // wants them to run while the peers are being mapped)
    if (h->world > 1) CUDA_TRY(cudaDeviceSynchronize());
    close_peers(h);
    const cudaIpcMemHandle_t *handles = static_cast<const cudaIpcMemHandle_t *>(all_ipc_handles);
    h->world = world;
    h->rank = rank;
    h->peers_are_ipc = true;
    for (uint32_t g = 0; g < world; ++g) {
        if (g == rank) {
            h->peer_t0[g] = h->graph.t0.get();
            h->peer_t1[g] = h->graph.t1.get();
            continue;
        }
        void *t0 = nullptr, *t1 = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&t0, handles[2 * g], cudaIpcMemLazyEnablePeerAccess);
        if (e == cudaSuccess) {
            h->peer_t0[g] = static_cast<float *>(t0);
            e = cudaIpcOpenMemHandle(&t1, handles[2 * g + 1], cudaIpcMemLazyEnablePeerAccess);
        }
        if (e != cudaSuccess) {
            close_peers(h);
            return fail(B2E_ERR_CUDA, std::string("cudaIpcOpenMemHandle (replica of rank ") + std::to_string(g) +
                                          "): " + cudaGetErrorString(e));
        }
        h->peer_t1[g] = static_cast<float *>(t1);
    }
    return B2E_OK;
}

extern "C" int b2e_exchange_open_local(b2e_handle *h, uint32_t world, uint32_t rank, b2e_handle *const *replicas) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (int rc = check_world(world, rank)) return rc;
    if (!replicas) return fail(B2E_ERR_INVALID, "null argument");
    CUDA_TRY(cudaDeviceSynchronize());
    close_peers(h);
    for (uint32_t g = 0; g < world; ++g) {
        const b2e_handle *r = g == rank ? h : replicas[g];
        if (!r || !r->graph.t0.get() || r->n != h->n || r->row_stride != h->row_stride)
            return fail(B2E_ERR_INVALID, "every replica must hold tables of the same shape");
        if (r->cfg.device != h->cfg.device) {
            int can = 0;
            CUDA_TRY(cudaDeviceCanAccessPeer(&can, h->cfg.device, r->cfg.device));
            if (!can) return fail(B2E_ERR_CUDA, "no peer access between the devices of the replicas");
            cudaError_t e = cudaDeviceEnablePeerAccess(r->cfg.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                return fail(B2E_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
            cudaGetLastError();
        }
    }
    h->world = world;
    h->rank = rank;
    for (uint32_t g = 0; g < world; ++g) {
        const b2e_handle *r = g == rank ? h : replicas[g];
        h->peer_t0[g] = r->graph.t0.get();
        h->peer_t1[g] = r->graph.t1.get();
    }
    return B2E_OK;
}

extern "C" int b2e_exchange_average(b2e_handle *h) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (h->world < 2) return B2E_OK;
    CUDA_TRY(launch_exchange_average(h->peer_t0, h->peer_t1, h->world, h->rank, h->n, h->row_stride,
                                     (h->cfg.embedding_size + 3u) / 4u, h->sm_count, h->train_stream));
    ++h->launches;
    return B2E_OK;
}

extern "C" int b2e_exchange_close(b2e_handle *h) {
    REQUIRE_HANDLE(h);
    CUDA_TRY(cudaDeviceSynchronize());
    close_peers(h);
    return B2E_OK;
}

extern "C" int b2e_tables_digest(b2e_handle *h, double *sums, uint64_t *words) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (!sums || !words) return fail(B2E_ERR_INVALID, "null argument");
    if (int rc = b2e_sync(h)) return rc;
    DeviceBuffer<> d_out;
    CUDA_TRY(d_out.reserve(56));
    CUDA_TRY(launch_tables_digest(h->graph.t0.get(), h->graph.t1.get(), h->n, h->row_stride, h->cfg.embedding_size,
                                  d_out.get(), h->sm_count, h->train_stream));
    unsigned char host[56];
    CUDA_TRY(cudaMemcpyAsync(host, d_out.get(), 56, cudaMemcpyDeviceToHost, h->train_stream));
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    ++h->launches;
    memcpy(sums, host, 32);
    memcpy(words, host + 32, 24);
    return B2E_OK;
}

// One table to the host without its row padding: packed on the device in slabs (train stream),
// each slab copied with one contiguous DMA (walk stream, idle here) while the next one is packed.
static int export_table(b2e_handle *h, const float *d_table, float *host) {
    const uint32_t dim = h->cfg.embedding_size;
    if (dim == h->row_stride) {
        CUDA_TRY(cudaMemcpyAsync(host, d_table, h->n * (uint64_t)dim * sizeof(float), cudaMemcpyDeviceToHost,
                                 h->train_stream));
        CUDA_TRY(cudaStreamSynchronize(h->train_stream));
        return B2E_OK;
    }
    const uint64_t slab_rows = std::max<uint64_t>(1, (256ull << 20) / (dim * sizeof(float)));
    struct Slabs {  // two staging buffers and their events, released on every way out
        DeviceBuffer<float> stage[2];
        cudaEvent_t packed[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
        ~Slabs() {
            for (cudaEvent_t event : {packed[0], packed[1], copied[0], copied[1]})
                if (event) cudaEventDestroy(event);
        }
    } s;
    for (int b = 0; b < 2; ++b) {
        CUDA_TRY(s.stage[b].reserve(std::min<uint64_t>(slab_rows, h->n) * dim * sizeof(float)));
        CUDA_TRY(cudaEventCreateWithFlags(&s.packed[b], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&s.copied[b], cudaEventDisableTiming));
    }
    uint64_t slab = 0;
    for (uint64_t row = 0; row < h->n; row += slab_rows, ++slab) {
        const int b = (int)(slab & 1);
        const uint64_t rows = std::min(slab_rows, h->n - row);
        if (slab >= 2) CUDA_TRY(cudaStreamWaitEvent(h->train_stream, s.copied[b], 0));  // the slab buffer is free again
        CUDA_TRY(launch_pack_rows(d_table + row * h->row_stride, rows, h->row_stride, dim, s.stage[b].get(),
                                  h->sm_count, h->train_stream));
        CUDA_TRY(cudaEventRecord(s.packed[b], h->train_stream));
        CUDA_TRY(cudaStreamWaitEvent(h->walk_stream, s.packed[b], 0));
        CUDA_TRY(cudaMemcpyAsync(host + row * dim, s.stage[b].get(), rows * dim * sizeof(float),
                                 cudaMemcpyDeviceToHost, h->walk_stream));
        CUDA_TRY(cudaEventRecord(s.copied[b], h->walk_stream));
        ++h->launches;
    }
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    return B2E_OK;
}

extern "C" int b2e_export_tables(b2e_handle *h, float *table0, float *table1) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (!table0 || !table1) return fail(B2E_ERR_INVALID, "null output buffer");
    if (int rc = b2e_sync(h)) return rc;
    if (int rc = export_table(h, h->graph.t0.get(), table0)) return rc;
    return export_table(h, h->graph.t1.get(), table1);
}

extern "C" int b2e_import_tables(b2e_handle *h, const float *table0, const float *table1) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (!table0 || !table1) return fail(B2E_ERR_INVALID, "null input buffer");
    if (int rc = b2e_sync(h)) return rc;
    const size_t width = h->cfg.embedding_size * sizeof(float);
    const size_t pitch = h->row_stride * sizeof(float);
    // the handle's streams are non-blocking: work on the legacy default stream is not ordered
    // with them, so everything here runs on the train stream and is waited for
    CUDA_TRY(cudaMemsetAsync(h->graph.t0.get(), 0, h->n * pitch, h->train_stream));
    CUDA_TRY(cudaMemsetAsync(h->graph.t1.get(), 0, h->n * pitch, h->train_stream));
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    CUDA_TRY(cudaMemcpy2DAsync(h->graph.t0.get(), pitch, table0, width, width, h->n, cudaMemcpyHostToDevice,
                               h->train_stream));
    CUDA_TRY(cudaMemcpy2DAsync(h->graph.t1.get(), pitch, table1, width, width, h->n, cudaMemcpyHostToDevice,
                               h->train_stream));
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    return B2E_OK;
}

extern "C" int b2e_export_alias(b2e_handle *h, uint32_t *threshold, uint32_t *alias) {
    if (!h || !threshold || !alias) return fail(B2E_ERR_INVALID, "null argument");
    if (!h->graph.alias.get()) return fail(B2E_ERR_STATE, "no alias table (uniform negatives or no graph)");
    if (h->h_alias_thr.empty()) {  // built on the device: fetched on demand (parity tests)
        CUDA_TRY(cudaSetDevice(h->cfg.device));
        std::vector<uint2> packed(h->n);
        CUDA_TRY(cudaMemcpy(packed.data(), h->graph.alias.get(), h->n * sizeof(uint2), cudaMemcpyDeviceToHost));
        h->h_alias_thr.resize(h->n);
        h->h_alias_idx.resize(h->n);
        for (uint64_t i = 0; i < h->n; ++i) {
            h->h_alias_thr[i] = packed[i].x;
            h->h_alias_idx[i] = packed[i].y;
        }
    }
    memcpy(threshold, h->h_alias_thr.data(), h->n * sizeof(uint32_t));
    memcpy(alias, h->h_alias_idx.data(), h->n * sizeof(uint32_t));
    return B2E_OK;
}

extern "C" int b2e_export_edge_alias(b2e_handle *h, uint32_t *table) {
    REQUIRE_HANDLE(h);
    if (!table) return fail(B2E_ERR_INVALID, "null argument");
    if (!h->graph.edge_alias.get()) return fail(B2E_ERR_STATE, "no edge alias table (unweighted graph or no graph)");
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    CUDA_TRY(cudaMemcpy(table, h->graph.edge_alias.get(), h->nnz * sizeof(uint2), cudaMemcpyDeviceToHost));
    return B2E_OK;
}

extern "C" int b2e_counters_read(b2e_handle *h, b2e_counters *out) {
    REQUIRE_HANDLE(h);
    if (!out) return fail(B2E_ERR_INVALID, "null argument");
    if (int rc = b2e_sync(h)) return rc;
    DeviceCounters c;
    CUDA_TRY(cudaMemcpyAsync(&c, h->d_counters.get(), sizeof(c), cudaMemcpyDeviceToHost, h->train_stream));
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    out->walk_steps = c.walk_steps;
    out->walk_trials = c.walk_trials;
    out->walk_searches = c.walk_searches;
    out->walk_probes = c.walk_probes;
    out->walk_filter_rejects = c.walk_filter_rejects;
    out->pairs = c.pairs;
    out->targets = c.targets;
    out->loss_sum = c.loss_sum;
    return B2E_OK;
}

extern "C" int b2e_counters_reset(b2e_handle *h) {
    REQUIRE_HANDLE(h);
    if (int rc = b2e_sync(h)) return rc;
    // not cudaMemset: the legacy default stream is not ordered with the non-blocking streams of
    // the handle, and a late memset would also clear the work counter of a running SGD kernel
    CUDA_TRY(cudaMemsetAsync(h->d_counters.get(), 0, sizeof(DeviceCounters), h->train_stream));
    CUDA_TRY(cudaStreamSynchronize(h->train_stream));
    return B2E_OK;
}

// ---- GloVe: co-occurrence of the walks, then one SGD pass over the triples ----
extern "C" int b2e_cooccurrence(b2e_handle *h, uint64_t seed, uint64_t first_walk, uint64_t n_walks,
                                uint64_t walk_id_stride, int accumulate, uint64_t *n_triples) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (walk_id_stride == 0) return fail(B2E_ERR_INVALID, "walk_id_stride must be positive");
    if (h->n_src == 0) return fail(B2E_ERR_INVALID, "the graph has no node with outgoing edges");
    if (int rc = b2e_sync(h)) return rc;
    const b2e_config &c = h->cfg;
    GloveState &g = h->graph.glove;
    if (!accumulate) { g.n_triples = 0; g.finalised = false; }
    std::string error;
    const uint64_t step = std::min<uint64_t>(h->chunk_cap, b2e::glove_chunk_walks(c.walk_length, c.window_size));
    for (uint64_t done = 0; done < n_walks; done += step) {
        const uint64_t count = std::min(step, n_walks - done);
        if (g.n_triples + 2ull * count * c.walk_length * c.window_size >= (1ull << 31))
            return fail(B2E_ERR_INVALID, "more than 2^31 co-occurrence entries in flight: lower walk_length, "
                                         "window_size or iterations");
        if (int rc = walk_into(h, seed, first_walk + done * walk_id_stride, count, walk_id_stride,
                               h->graph.walks[0].get(), h->walk_stream))
            return rc;
        if (glove_accumulate(g, h->graph.walks[0].get(), count, c.walk_length, c.window_size, h->walk_stream, error))
            return fail(B2E_ERR_CUDA, error);
        h->launches += 2;
    }
    if (glove_finalise(g, h->n, h->walk_stream, error)) return fail(B2E_ERR_CUDA, error);
    ++h->launches;
    if (n_triples) *n_triples = g.n_triples;
    return B2E_OK;
}

extern "C" int b2e_cooccurrence_export(b2e_handle *h, uint32_t *centre, uint32_t *context, uint32_t *count) {
    REQUIRE_HANDLE(h);
    if (!centre || !context || !count) return fail(B2E_ERR_INVALID, "null output buffer");
    if (int rc = b2e_sync(h)) return rc;
    const uint64_t m = h->graph.glove.n_triples;
    std::vector<unsigned long long> keys(m);
    CUDA_TRY(cudaMemcpyAsync(keys.data(), h->graph.glove.d_keys.get(), m * sizeof(unsigned long long),
                             cudaMemcpyDeviceToHost, h->walk_stream));
    CUDA_TRY(cudaMemcpyAsync(count, h->graph.glove.d_counts.get(), m * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                             h->walk_stream));
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    for (uint64_t i = 0; i < m; ++i) {
        centre[i] = (uint32_t)(keys[i] >> 32);
        context[i] = (uint32_t)keys[i];
    }
    return B2E_OK;
}

extern "C" int b2e_glove_train(b2e_handle *h, float learning_rate) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (h->cfg.model != B2E_GLOVE) return fail(B2E_ERR_STATE, "the handle was not created for GloVe");
    if (!h->graph.glove.finalised) return fail(B2E_ERR_STATE, "b2e_cooccurrence must be called first");
    const b2e_config &c = h->cfg;
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    // centres in flight: like SkipGram, about one per 16 nodes on small graphs (staleness)
    const uint64_t max_warps = c.max_concurrent_walks ? c.max_concurrent_walks
                                                       : std::max<uint64_t>(16, h->n / 16);
    CUDA_TRY(glove_train(h->graph.glove, h->n, h->row_stride, c.embedding_size, c.glove_alpha, c.clipping_value,
                              learning_rate, h->graph.t0.get(), h->graph.t1.get(), h->d_counters.get(), c.deterministic != 0,
                              h->sm_count, max_warps, h->train_stream));
    if (h->graph.glove.n_triples) ++h->launches;
    return B2E_OK;
}

// ---- GloVe by centre range (glove.cu, "co-occurrence by centre range") ----
// An epoch whose co-occurrence exceeds one sort is walked whole, its token positions are bucketed
// by range of centre id, and the ranges are counted and trained one by one in ascending order of
// centre.  x_max is the largest count of the WHOLE epoch, so with more than one range the ranges
// are counted twice: once for x_max, once to train.  The same steps make the sharded epoch of
// several GPUs: every rank walks the whole epoch, then counts and trains only the centres it owns.

// the walks of a whole epoch into HBM, and their token histogram (host copy in g.histogram)
static int glove_walk_epoch(b2e_handle *h, uint64_t seed, uint64_t first_walk, uint64_t per_epoch) {
    GloveState &g = h->graph.glove;
    const uint32_t L = h->cfg.walk_length;
    const uint64_t tokens = per_epoch * L;
    g.histogram.clear();
    CUDA_TRY(g.d_epoch_walks.reserve(tokens * sizeof(uint32_t)));
    CUDA_TRY(g.d_histogram.reserve(h->n * sizeof(uint32_t)));
    for (uint64_t done = 0; done < per_epoch; done += h->chunk_cap) {
        const uint64_t count = std::min(h->chunk_cap, per_epoch - done);
        if (int rc = walk_into(h, seed, first_walk + done, count, 1, g.d_epoch_walks.get() + done * L, h->walk_stream)) return rc;
    }
    CUDA_TRY(glove_token_histogram(g.d_epoch_walks.get(), tokens, g.d_histogram.get(), h->n, h->walk_stream));
    std::vector<uint32_t> histogram(h->n);
    CUDA_TRY(cudaMemcpyAsync(histogram.data(), g.d_histogram.get(), h->n * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                             h->walk_stream));
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    h->launches += 2;
    g.histogram.swap(histogram);
    g.epoch_tokens = tokens;
    return B2E_OK;
}

// Cut the centres [lo, hi) into ranges holding at most capacity_slots key slots each (one node
// may exceed it) and bucket the positions of their tokens by range (tokens of other centres are
// skipped).
static int glove_bucket_ranges(b2e_handle *h, uint32_t lo, uint32_t hi, uint64_t capacity_slots) {
    GloveState &g = h->graph.glove;
    const uint32_t W = h->cfg.window_size;
    std::vector<uint32_t> bounds(1, lo);
    std::vector<unsigned long long> offsets(1, 0ull);
    uint64_t in_range = 0, placed = 0;
    for (uint64_t v = lo; v < hi; ++v) {
        const uint64_t slots = (uint64_t)g.histogram[v] * 2ull * W;
        if (in_range && in_range + slots > capacity_slots) {
            bounds.push_back((uint32_t)v);
            offsets.push_back(placed);
            in_range = 0;
        }
        in_range += slots;
        placed += g.histogram[v];
        if (slots >= (1ull << 31))
            return fail(B2E_ERR_INVALID, "one node alone has 2^31 co-occurrence slots in an epoch: lower walk_length, "
                                         "window_size or iterations");
    }
    bounds.push_back(hi);
    offsets.push_back(placed);
    const uint32_t ranges = (uint32_t)bounds.size() - 1u;
    g.last_ranges = ranges;
    g.range_kept = false;
    CUDA_TRY(g.d_bounds.reserve(bounds.size() * sizeof(uint32_t)));
    CUDA_TRY(g.d_cursor.reserve(ranges * sizeof(unsigned long long)));
    CUDA_TRY(g.d_positions.reserve(std::max<uint64_t>(placed, 1) * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemcpyAsync(g.d_bounds.get(), bounds.data(), bounds.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, h->walk_stream));
    CUDA_TRY(cudaMemcpyAsync(g.d_cursor.get(), offsets.data(), ranges * sizeof(unsigned long long), cudaMemcpyHostToDevice, h->walk_stream));
    CUDA_TRY(glove_bucket_positions(g.d_epoch_walks.get(), g.epoch_tokens, g.d_bounds.get(), ranges, g.d_cursor.get(), g.d_positions.get(),
                                    h->walk_stream));
    CUDA_TRY(cudaStreamSynchronize(h->walk_stream));
    ++h->launches;
    g.range_bounds.swap(bounds);
    g.range_offsets.swap(offsets);
    return B2E_OK;
}

static int glove_count_range(b2e_handle *h, uint32_t r) {
    GloveState &g = h->graph.glove;
    std::string error;
    if (glove_range_triples(g, g.d_epoch_walks.get(), h->cfg.walk_length, h->cfg.window_size,
                            g.d_positions.get() + g.range_offsets[r], g.range_offsets[r + 1] - g.range_offsets[r],
                            h->walk_stream, error))
        return fail(B2E_ERR_CUDA, error);
    h->launches += 2;
    return B2E_OK;
}

// the largest count of the bucketed ranges (0 without triples); a single range keeps its triples
static int glove_count_ranges(b2e_handle *h, uint32_t *largest) {
    GloveState &g = h->graph.glove;
    const uint32_t ranges = (uint32_t)g.range_bounds.size() - 1u;
    *largest = 0;
    std::string error;
    for (uint32_t r = 0; r < ranges; ++r) {
        if (int rc = glove_count_range(h, r)) return rc;
        uint32_t local = 0;
        if (glove_max_count(g, &local, h->walk_stream, error)) return fail(B2E_ERR_CUDA, error);
        *largest = std::max(*largest, local);
    }
    g.range_kept = ranges == 1;
    return B2E_OK;
}

// one SGD pass over the bucketed ranges in ascending order of centre, weights against x_max
static int glove_train_ranges(b2e_handle *h, float lr, uint32_t x_max) {
    GloveState &g = h->graph.glove;
    const uint32_t ranges = (uint32_t)g.range_bounds.size() - 1u;
    std::string error;
    for (uint32_t r = 0; r < ranges; ++r) {
        if (!g.range_kept)
            if (int rc = glove_count_range(h, r)) return rc;
        if (g.n_triples == 0) continue;
        if (glove_finalise(g, h->n, h->walk_stream, error)) return fail(B2E_ERR_CUDA, error);
        g.max_count = x_max;
        if (int rc = b2e_glove_train(h, lr)) return rc;
        CUDA_TRY(cudaStreamSynchronize(h->train_stream));  // the triples are replaced by the next range
    }
    g.range_kept = false;
    return B2E_OK;
}

// key slots one sort may hold (B2E_GLOVE_SLOTS overrides: tests force many ranges on small graphs)
static uint64_t glove_capacity_slots() {
    if (const char *env = getenv("B2E_GLOVE_SLOTS")) return std::max<uint64_t>(64, strtoull(env, nullptr, 10));
    return 1ull << 28;
}

static int glove_epoch_by_ranges(b2e_handle *h, uint64_t seed, uint64_t first_walk, uint64_t per_epoch, float lr,
                                 uint64_t capacity_slots) {
    if (int rc = glove_walk_epoch(h, seed, first_walk, per_epoch)) return rc;
    if (int rc = glove_bucket_ranges(h, 0, (uint32_t)h->n, capacity_slots)) return rc;
    uint32_t x_max = 0;
    if (int rc = glove_count_ranges(h, &x_max)) return rc;
    return glove_train_ranges(h, lr, x_max);
}

// Owners of a sharded epoch: with S the key slots of the epoch (2 W per token) and c_v the slots
// of the nodes before v, rank r owns the nodes with r S / G <= c_v < (r + 1) S / G; nodes past the
// last slot go to the last rank.  A pure function of the histogram: every rank finds the same bounds.
static void glove_owner_bounds(const std::vector<uint32_t> &histogram, uint32_t W, uint32_t world, uint32_t *bounds) {
    const uint64_t n = histogram.size();
    uint64_t total = 0;
    for (const uint32_t tokens : histogram) total += (uint64_t)tokens * 2ull * W;
    bounds[0] = 0;
    uint32_t r = 1;
    uint64_t before = 0;
    for (uint64_t v = 0; v < n && r < world; ++v) {
        while (r < world && before * world >= r * total) bounds[r++] = (uint32_t)v;
        before += (uint64_t)histogram[v] * 2ull * W;
    }
    while (r <= world) bounds[r++] = (uint32_t)n;
}

static int require_glove(b2e_handle *h) {
    if (int rc = require_graph(h)) return rc;
    if (h->cfg.model != B2E_GLOVE) return fail(B2E_ERR_STATE, "the handle was not created for GloVe");
    return B2E_OK;
}

extern "C" int b2e_glove_walk_epoch(b2e_handle *h, uint64_t seed, uint64_t first_walk, uint64_t n_walks) {
    REQUIRE_HANDLE(h);
    if (int rc = require_glove(h)) return rc;
    if (h->n_src == 0) return fail(B2E_ERR_INVALID, "the graph has no node with outgoing edges");
    if (int rc = b2e_sync(h)) return rc;
    return glove_walk_epoch(h, seed, first_walk, n_walks);
}

extern "C" int b2e_glove_shard_count(b2e_handle *h, uint32_t world, uint32_t rank, uint32_t *owner_bounds,
                                     uint32_t *local_max) {
    REQUIRE_HANDLE(h);
    if (int rc = require_glove(h)) return rc;
    if (int rc = check_world(world, rank)) return rc;
    if (!local_max) return fail(B2E_ERR_INVALID, "null argument");
    GloveState &g = h->graph.glove;
    if (g.histogram.size() != h->n) return fail(B2E_ERR_STATE, "b2e_glove_walk_epoch must be called first");
    if (int rc = b2e_sync(h)) return rc;
    glove_owner_bounds(g.histogram, h->cfg.window_size, world, g.owner_bounds);
    g.owner_world = world;
    if (owner_bounds) memcpy(owner_bounds, g.owner_bounds, (world + 1) * sizeof(uint32_t));
    if (int rc = glove_bucket_ranges(h, g.owner_bounds[rank], g.owner_bounds[rank + 1], glove_capacity_slots())) return rc;
    return glove_count_ranges(h, local_max);
}

extern "C" int b2e_glove_shard_train(b2e_handle *h, float learning_rate, uint32_t max_count) {
    REQUIRE_HANDLE(h);
    if (int rc = require_glove(h)) return rc;
    GloveState &g = h->graph.glove;
    if (g.owner_world == 0 || g.range_bounds.empty())
        return fail(B2E_ERR_STATE, "b2e_glove_shard_count must be called first");
    if (g.owner_world > 1) {  // the base of the merge: T1 before this epoch's training (same stream, ordered)
        const size_t bytes = h->n * (size_t)h->row_stride * sizeof(float);
        CUDA_TRY(g.d_t1_snapshot.reserve(bytes));
        CUDA_TRY(cudaMemcpyAsync(g.d_t1_snapshot.get(), h->graph.t1.get(), bytes, cudaMemcpyDeviceToDevice, h->train_stream));
    }
    const int rc = glove_train_ranges(h, learning_rate, std::max(max_count, 1u));
    g.range_bounds.clear();  // trained: the next epoch counts anew
    return rc;
}

extern "C" int b2e_glove_merge(b2e_handle *h) {
    REQUIRE_HANDLE(h);
    if (int rc = require_glove(h)) return rc;
    if (h->world < 2) return B2E_OK;
    GloveState &g = h->graph.glove;
    if (g.owner_world != h->world || !g.d_t1_snapshot.get())
        return fail(B2E_ERR_STATE, "b2e_glove_shard_count and b2e_glove_shard_train with the world of the exchange "
                                   "must come first");
    CUDA_TRY(launch_glove_merge(h->peer_t0, h->peer_t1, g.d_t1_snapshot.get(), g.owner_bounds, h->world, h->rank, h->n,
                                h->row_stride, (h->cfg.embedding_size + 3u) / 4u, h->sm_count, h->train_stream));
    ++h->launches;
    return B2E_OK;
}

static int fit_glove(b2e_handle *h, uint64_t seed, float *table0, float *table1, float *epoch_loss) {
    const b2e_config &c = h->cfg;
    if (int rc = b2e_init_tables(h, seed)) return rc;
    const uint64_t per_epoch = (uint64_t)c.iterations * h->n_src;
    const uint64_t capacity = glove_capacity_slots();
    const bool by_ranges = 2ull * per_epoch * c.walk_length * c.window_size > capacity;
    float lr = c.learning_rate;
    for (uint32_t epoch = 0; epoch < c.epochs; ++epoch) {
        if (int rc = b2e_counters_reset(h)) return rc;
        if (by_ranges) {
            if (int rc = glove_epoch_by_ranges(h, seed, (uint64_t)epoch * per_epoch, per_epoch, lr, capacity)) return rc;
        } else {
            if (int rc = b2e_cooccurrence(h, seed, (uint64_t)epoch * per_epoch, per_epoch, 1, 0, nullptr)) return rc;
            if (int rc = b2e_glove_train(h, lr)) return rc;
        }
        b2e_counters counters;
        if (int rc = b2e_counters_read(h, &counters)) return rc;
        if (epoch_loss) epoch_loss[epoch] = counters.pairs ? (float)(counters.loss_sum / (double)counters.pairs) : 0.0f;
        lr = lr * c.learning_rate_decay;
    }
    return b2e_export_tables(h, table0, table1);
}

// The whole path: init, then per epoch walk chunk k+1 on the walk stream while the SGD
// kernel consumes chunk k on the train stream (two walk buffers, event-ordered).
extern "C" int b2e_fit(b2e_handle *h, uint64_t seed, float *table0, float *table1, float *epoch_loss) {
    REQUIRE_HANDLE(h);
    if (int rc = require_graph(h)) return rc;
    if (!table0 || !table1) return fail(B2E_ERR_INVALID, "null output buffer");
    if (h->n_src == 0) return fail(B2E_ERR_INVALID, "the graph has no node with outgoing edges");
    const b2e_config &c = h->cfg;
    if (c.model == B2E_GLOVE) return fit_glove(h, seed, table0, table1, epoch_loss);
    if (int rc = b2e_init_tables(h, seed)) return rc;
    const uint64_t per_epoch = (uint64_t)c.iterations * h->n_src;
    float lr = c.learning_rate;
    uint64_t chunk_index = 0;
    for (uint32_t epoch = 0; epoch < c.epochs; ++epoch) {
        if (int rc = b2e_counters_reset(h)) return rc;
        const uint64_t base = (uint64_t)epoch * per_epoch;
        uint64_t issued = 0;
        // prime the pipeline with the first chunk, then keep one walk chunk ahead of the SGD
        uint64_t count = std::min(h->chunk_cap, per_epoch);
        if (int rc = b2e_walk_chunk(h, seed, base, count, 1, chunk_index & 1)) return rc;
        issued = count;
        while (true) {
            const uint32_t slot = chunk_index & 1;
            if (issued < per_epoch) {
                const uint64_t next = std::min(h->chunk_cap, per_epoch - issued);
                if (int rc = b2e_walk_chunk(h, seed, base + issued, next, 1, slot ^ 1)) return rc;
                issued += next;
                if (int rc = b2e_train_chunk(h, seed, slot, lr)) return rc;
                ++chunk_index;
            } else {
                if (int rc = b2e_train_chunk(h, seed, slot, lr)) return rc;
                ++chunk_index;
                break;
            }
        }
        b2e_counters counters;
        if (int rc = b2e_counters_read(h, &counters)) return rc;
        if (epoch_loss) epoch_loss[epoch] = counters.pairs ? (float)(counters.loss_sum / (double)counters.pairs) : 0.0f;
        lr = lr * c.learning_rate_decay;
    }
    // role order of the reference: [central, contextual]; for CBOW the table scored against
    // the centre node is the output table
    if (c.model == B2E_CBOW) return b2e_export_tables(h, table1, table0);
    return b2e_export_tables(h, table0, table1);
}

// ---- resident graphs: built on the GPU, handed to a handle without leaving HBM ----
// a host CSR uploaded once, to be shared by several handles (b2e_load_graph checks its contents)
extern "C" int b2e_graph_from_csr(int device, const int64_t *indptr, const uint32_t *indices, uint64_t n,
                                  uint64_t nnz, b2e_graph **out) {
    return b2e_graph_from_csr_weighted(device, indptr, indices, nullptr, n, nnz, out);
}

extern "C" int b2e_graph_from_csr_weighted(int device, const int64_t *indptr, const uint32_t *indices,
                                           const float *weights, uint64_t n, uint64_t nnz, b2e_graph **out) {
    if (!out || !indptr || (!indices && nnz)) return fail(B2E_ERR_INVALID, "null argument");
    if (n == 0 || n >= 0xFFFFFF00ull) return fail(B2E_ERR_INVALID, "the number of nodes must be in [1, 0xFFFFFF00)");
    if (indptr[0] != 0 || (uint64_t)indptr[n] != nnz)
        return fail(B2E_ERR_INVALID, "indptr must start at 0 and end at nnz");
    for (uint64_t v = 0; v < n; ++v)
        if (indptr[v + 1] < indptr[v]) return fail(B2E_ERR_INVALID, "indptr must be non-decreasing");
    if (weights)
        for (uint64_t e = 0; e < nnz; ++e)
            if (!(weights[e] >= 0.0f)) return fail(B2E_ERR_INVALID, "edge weights must be non-negative numbers");
    if (int rc = select_device(device)) return rc;
    std::unique_ptr<b2e_graph, GraphRelease> g(new (std::nothrow) b2e_graph());
    if (!g) return fail(B2E_ERR_INVALID, "out of host memory");
    g->device = device;
    g->csr.n = n;
    g->csr.nnz = nnz;
    CUDA_TRY(g->csr.indptr.reserve((n + 1) * sizeof(int64_t)));
    CUDA_TRY(g->csr.indices.reserve(std::max<uint64_t>(nnz, 1) * sizeof(uint32_t)));
    CUDA_TRY(cudaMemcpy(g->csr.indptr.get(), indptr, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice));
    if (nnz) CUDA_TRY(cudaMemcpy(g->csr.indices.get(), indices, nnz * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (weights) {
        CUDA_TRY(g->csr.weights.reserve(std::max<uint64_t>(nnz, 1) * sizeof(float)));
        if (nnz) CUDA_TRY(cudaMemcpy(g->csr.weights.get(), weights, nnz * sizeof(float), cudaMemcpyHostToDevice));
    }
    *out = g.release();
    return B2E_OK;
}

extern "C" int b2e_graph_shape(const b2e_graph *g, uint64_t *n, uint64_t *nnz) {
    if (!g || !n || !nnz) return fail(B2E_ERR_INVALID, "null argument");
    *n = g->csr.n;
    *nnz = g->csr.nnz;
    return B2E_OK;
}

extern "C" int b2e_graph_export(const b2e_graph *g, int64_t *indptr, uint32_t *indices) {
    if (!g || !indptr || (!indices && g->csr.nnz)) return fail(B2E_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(g->device));
    CUDA_TRY(cudaMemcpy(indptr, g->csr.indptr.get(), (g->csr.n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost));
    if (g->csr.nnz)
        CUDA_TRY(cudaMemcpy(indices, g->csr.indices.get(), g->csr.nnz * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return B2E_OK;
}

extern "C" int b2e_graph_weighted(const b2e_graph *g) { return g && g->csr.weights.get() ? 1 : 0; }

extern "C" int b2e_graph_export_weights(const b2e_graph *g, float *weights) {
    if (!g || (!weights && g->csr.nnz)) return fail(B2E_ERR_INVALID, "null argument");
    if (!g->csr.weights.get()) return fail(B2E_ERR_STATE, "the graph has no edge weights");
    CUDA_TRY(cudaSetDevice(g->device));
    if (g->csr.nnz)
        CUDA_TRY(cudaMemcpy(weights, g->csr.weights.get(), g->csr.nnz * sizeof(float), cudaMemcpyDeviceToHost));
    return B2E_OK;
}

extern "C" void b2e_graph_destroy(b2e_graph *g) {
    if (!g) return;
    cudaSetDevice(g->device);
    release_graph(g);
}

extern "C" int b2e_load_graph(b2e_handle *h, b2e_graph *g) {
    REQUIRE_HANDLE(h);
    if (!g) return fail(B2E_ERR_INVALID, "null graph");
    if (g->device != h->cfg.device) return fail(B2E_ERR_INVALID, "the graph lives on another device than the handle");
    if (g->csr.n == 0) return fail(B2E_ERR_INVALID, "The provided graph is empty.");
    if (g->csr.nnz == 0) return fail(B2E_ERR_INVALID, "The provided graph does not have edges.");
    // nothing comes back to the host: start nodes, alias table, edge alias tables (a weighted
    // graph, normalize_by_degree), filters are all built from the resident arrays (an exponent
    // without an exact form fetches the offsets, see alias_build.cu)
    std::vector<int64_t> indptr;
    const double alpha = (double)h->cfg.negative_sampling_exponent;
    if (h->cfg.use_scale_free_distribution && alpha != 0.0 && alpha != 0.5 && alpha != 0.75 && alpha != 1.0) {
        indptr.resize(g->csr.n + 1);
        CUDA_TRY(cudaMemcpy(indptr.data(), g->csr.indptr.get(), indptr.size() * sizeof(int64_t), cudaMemcpyDeviceToHost));
    }
    ++g->references;  // keep it alive across drop_graph() of a handle that already walks on it
    const int rc = load_graph_common(h, indptr.empty() ? nullptr : indptr.data(), nullptr, nullptr, g->csr.n,
                                     g->csr.nnz, g);
    release_graph(g);
    return rc;
}

// ---- graph ingest (csrc/graph_build.cu) ----
// the status of an ingest call: cudaErrorInvalidValue marks bad input, named in `error`
static int ingest_status(cudaError_t e, const std::string &error) {
    if (e == cudaErrorInvalidValue) return fail(B2E_ERR_INVALID, error);
    if (e != cudaSuccess) return fail(B2E_ERR_CUDA, error);
    return B2E_OK;
}

static int deliver_graph(int device, cudaError_t e, const std::string &error, ResidentCsr &csr, b2e_graph **out) {
    if (int rc = ingest_status(e, error)) return rc;
    b2e_graph *g = new (std::nothrow) b2e_graph();
    if (!g) return fail(B2E_ERR_INVALID, "out of host memory");
    g->csr = std::move(csr);
    g->device = device;
    *out = g;
    return B2E_OK;
}

// the checks b2e_graph_from_edges and b2e_csr_from_edges share, after their own output arguments
static int check_edges(const uint32_t *src, const uint32_t *dst, uint64_t n_edges, uint64_t n_nodes) {
    if (n_edges && (!src || !dst)) return fail(B2E_ERR_INVALID, "null argument");
    if (n_nodes == 0 || n_nodes >= 0xFFFFFF00ull)
        return fail(B2E_ERR_INVALID, "the number of nodes must be in [1, 0xFFFFFF00)");
    return B2E_OK;
}

// the checks b2e_graph_synthetic and b2e_synthetic_csr share, after their own output arguments
static int check_synthetic(int kind, uint64_t n_nodes, uint32_t scale, uint64_t n_edges) {
    if (kind != 0 && kind != 1) return fail(B2E_ERR_INVALID, "kind must be 0 (Erdos-Renyi) or 1 (R-MAT)");
    if (n_nodes < 2 || n_nodes >= 0xFFFFFF00ull)
        return fail(B2E_ERR_INVALID, "the number of nodes must be in [2, 0xFFFFFF00)");
    if (kind == 1 && (scale == 0 || scale > 32 || (scale < 32 && n_nodes > (1ull << scale))))
        return fail(B2E_ERR_INVALID, "R-MAT needs 1 <= scale <= 32 and n_nodes <= 2^scale");
    if ((double)n_edges > 0.5 * (double)n_nodes * (double)(n_nodes - 1) * 0.5)
        return fail(B2E_ERR_INVALID, "Too many edges requested.");
    return B2E_OK;
}

extern "C" int b2e_graph_from_edges(int device, const uint32_t *src, const uint32_t *dst, uint64_t n_edges,
                                    uint64_t n_nodes, int symmetrise, b2e_graph **out) {
    return b2e_graph_from_edges_weighted(device, src, dst, nullptr, n_edges, n_nodes, symmetrise, out);
}

extern "C" int b2e_graph_from_edges_weighted(int device, const uint32_t *src, const uint32_t *dst,
                                             const float *weights, uint64_t n_edges, uint64_t n_nodes, int symmetrise,
                                             b2e_graph **out) {
    if (!out) return fail(B2E_ERR_INVALID, "null argument");
    if (int rc = check_edges(src, dst, n_edges, n_nodes)) return rc;
    if (int rc = select_device(device)) return rc;
    std::string error;
    ResidentCsr csr;
    uint64_t nnz = 0;
    cudaError_t e = csr_from_edges(src, dst, weights, n_edges, n_nodes, symmetrise, nullptr, nullptr, nullptr, 0, &nnz,
                                   error, &csr);
    return deliver_graph(device, e, error, csr, out);
}

extern "C" int b2e_graph_synthetic(int device, int kind, uint64_t n_nodes, uint32_t scale, uint64_t n_edges,
                                   uint64_t seed, uint64_t t_a, uint64_t t_ab, uint64_t t_abc, b2e_graph **out) {
    if (!out) return fail(B2E_ERR_INVALID, "null argument");
    if (int rc = check_synthetic(kind, n_nodes, scale, n_edges)) return rc;
    if (int rc = select_device(device)) return rc;
    std::string error;
    ResidentCsr csr;
    uint64_t nnz = 0;
    cudaError_t e = synthetic_csr(kind, n_nodes, scale, n_edges, seed, t_a, t_ab, t_abc, nullptr, nullptr, 0, &nnz,
                                  error, &csr);
    return deliver_graph(device, e, error, csr, out);
}

extern "C" int b2e_csr_from_edges(int device, const uint32_t *src, const uint32_t *dst, uint64_t n_edges,
                                  uint64_t n_nodes, int symmetrise, int64_t *indptr, uint32_t *indices,
                                  uint64_t indices_capacity, uint64_t *nnz) {
    return b2e_csr_from_edges_weighted(device, src, dst, nullptr, n_edges, n_nodes, symmetrise, indptr, indices,
                                       nullptr, indices_capacity, nnz);
}

extern "C" int b2e_csr_from_edges_weighted(int device, const uint32_t *src, const uint32_t *dst,
                                           const float *weights, uint64_t n_edges, uint64_t n_nodes, int symmetrise,
                                           int64_t *indptr, uint32_t *indices, float *out_weights,
                                           uint64_t indices_capacity, uint64_t *nnz) {
    if (!indptr || !nnz || (n_edges && !indices) || (n_edges && weights && !out_weights))
        return fail(B2E_ERR_INVALID, "null argument");
    if (int rc = check_edges(src, dst, n_edges, n_nodes)) return rc;
    if (int rc = select_device(device)) return rc;
    std::string error;
    cudaError_t e = csr_from_edges(src, dst, weights, n_edges, n_nodes, symmetrise, indptr, indices, out_weights,
                                   indices_capacity, nnz, error);
    return ingest_status(e, error);
}

extern "C" int b2e_synthetic_csr(int device, int kind, uint64_t n_nodes, uint32_t scale, uint64_t n_edges,
                                 uint64_t seed, uint64_t t_a, uint64_t t_ab, uint64_t t_abc,
                                 int64_t *indptr, uint32_t *indices, uint64_t indices_capacity,
                                 uint64_t *nnz) {
    if (!indptr || !indices || !nnz) return fail(B2E_ERR_INVALID, "null argument");
    if (int rc = check_synthetic(kind, n_nodes, scale, n_edges)) return rc;
    if (indices_capacity < 2 * n_edges) return fail(B2E_ERR_INVALID, "indices_capacity must be >= 2 * n_edges");
    if (int rc = select_device(device)) return rc;
    std::string error;
    cudaError_t e = synthetic_csr(kind, n_nodes, scale, n_edges, seed, t_a, t_ab, t_abc, indptr, indices,
                                  indices_capacity, nnz, error);
    return ingest_status(e, error);
}
