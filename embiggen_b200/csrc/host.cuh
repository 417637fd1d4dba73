// Host side of the C ABI: the owner of device memory, the error slot, device selection and the
// handle layout.  Kernels do not need any of it.
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "common.cuh"

namespace b2e {

// One cudaMalloc allocation, freed by the destructor.  reserve() only grows: a larger request
// frees the old allocation first, then allocates.
template <typename T = void>
class DeviceBuffer {
public:
    DeviceBuffer() = default;
    DeviceBuffer(DeviceBuffer &&other) noexcept { *this = std::move(other); }
    DeviceBuffer &operator=(DeviceBuffer &&other) noexcept {
        if (this != &other) {
            reset();
            std::swap(ptr_, other.ptr_);
            std::swap(bytes_, other.bytes_);
        }
        return *this;
    }
    DeviceBuffer(const DeviceBuffer &) = delete;
    DeviceBuffer &operator=(const DeviceBuffer &) = delete;
    ~DeviceBuffer() { cudaFree(ptr_); }

    T *get() const { return ptr_; }
    size_t bytes() const { return bytes_; }
    cudaError_t reserve(size_t want) {
        if (want <= bytes_) return cudaSuccess;
        reset();
        void *p = nullptr;
        const cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) {
            ptr_ = static_cast<T *>(p);
            bytes_ = want;
        }
        return e;
    }
    void reset() {
        cudaFree(ptr_);
        ptr_ = nullptr;
        bytes_ = 0;
    }

private:
    T *ptr_ = nullptr;
    size_t bytes_ = 0;
};

// the message b2e_last_error() returns: the last failure of this thread
inline thread_local std::string g_last_error;

inline int fail(int status, const std::string &message) {
    g_last_error = message;
    return status;
}

// in a function that returns a b2e_status
#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess)                                                               \
            return b2e::fail(B2E_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

// in an internal function that returns a cudaError_t and names the failure in `error`
#define CUDA_CHECK(expr)                                                 \
    do {                                                                 \
        cudaError_t _e = (expr);                                         \
        if (_e != cudaSuccess) {                                         \
            error = std::string(#expr) + ": " + cudaGetErrorString(_e);  \
            return _e;                                                   \
        }                                                                \
    } while (0)

// there is a device, `device` is one of them, and it is now current
inline int select_device(int device) {
    int count = 0;
    const cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(B2E_ERR_CUDA, std::string("no CUDA device available (there is no CPU fallback): ") +
                                      cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail(B2E_ERR_INVALID, "device ordinal out of range");
    CUDA_TRY(cudaSetDevice(device));
    return B2E_OK;
}

// GloVe (glove.cu): the co-occurrence triples of an epoch, sorted by (centre << 32 | context)
struct GloveState {
    DeviceBuffer<unsigned long long> d_keys;
    DeviceBuffer<uint32_t> d_counts;
    DeviceBuffer<uint64_t> d_rowptr;
    uint64_t n_triples = 0;
    uint32_t max_count = 1;
    bool finalised = false;
    DeviceBuffer<unsigned long long> d_scratch_keys, d_merge_keys;
    DeviceBuffer<uint32_t> d_merge_counts;
    DeviceBuffer<> d_temp, d_scalar;
    // co-occurrence by centre range: the walks of an epoch, their token positions bucketed by range
    DeviceBuffer<uint32_t> d_epoch_walks, d_histogram, d_bounds;
    DeviceBuffer<unsigned long long> d_positions, d_cursor;
    uint32_t last_ranges = 0;  // how many centre ranges the last epoch took (1 = one piece)
    uint64_t epoch_tokens = 0;                    // tokens of the walked epoch (d_epoch_walks)
    std::vector<uint32_t> histogram;              // tokens per node of the walked epoch (host copy)
    std::vector<uint32_t> range_bounds;           // range r: range_bounds[r] <= centre < range_bounds[r + 1]
    std::vector<unsigned long long> range_offsets;  // bucketed occurrences before range r
    bool range_kept = false;                      // one range: its triples are resident, counted once
    // sharded epoch (several GPUs): rank r owns the centres [owner_bounds[r], owner_bounds[r + 1])
    uint32_t owner_world = 0, owner_bounds[B2E_MAX_WORLD + 1] = {0};
    DeviceBuffer<float> d_t1_snapshot;  // T1 as it stood before this epoch's training (the merge's base)
};
uint64_t glove_chunk_walks(uint32_t walk_length, uint32_t window);
cudaError_t glove_accumulate(GloveState &g, const uint32_t *d_walks, uint64_t n_walks, uint32_t walk_length,
                             uint32_t window, cudaStream_t stream, std::string &error);
cudaError_t glove_finalise(GloveState &g, uint64_t n, cudaStream_t stream, std::string &error);
cudaError_t glove_train(const GloveState &g, uint64_t n, uint32_t row_stride, uint32_t embedding_size,
                        float alpha, float clip, float lr, float *t0, float *t1, DeviceCounters *counters,
                        bool deterministic, int sm_count, uint64_t max_warps, cudaStream_t stream);
// co-occurrence by centre range (glove.cu): histogram of the epoch's tokens, occurrences bucketed
// by range, the triples of one range
cudaError_t glove_token_histogram(const uint32_t *d_walks, uint64_t tokens, uint32_t *d_histogram, uint64_t n,
                                  cudaStream_t stream);
cudaError_t glove_bucket_positions(const uint32_t *d_walks, uint64_t tokens, const uint32_t *d_bounds, uint32_t ranges,
                                   unsigned long long *d_cursor, unsigned long long *d_positions,
                                   cudaStream_t stream);
cudaError_t glove_range_triples(GloveState &g, const uint32_t *d_walks, uint32_t L, uint32_t W,
                                const unsigned long long *d_positions, uint64_t count, cudaStream_t stream,
                                std::string &error);
cudaError_t glove_max_count(GloveState &g, uint32_t *max_count, cudaStream_t stream, std::string &error);

// a CSR that stays in HBM (b2e_graph): built by graph_build.cu, or uploaded by b2e_load_csr*
struct ResidentCsr {
    DeviceBuffer<int64_t> indptr;
    DeviceBuffer<uint32_t> indices;
    DeviceBuffer<float> weights;  // one per edge, never negative; empty for an unweighted graph
    uint64_t n = 0, nnz = 0;
};
// `resident` != nullptr: the device arrays move into it and the host buffers are not touched.
// `weights` (nullable, one per input edge) makes a weighted graph; `out_weights` receives its nnz
// weights when the CSR goes to host buffers.
cudaError_t csr_from_edges(const uint32_t *src, const uint32_t *dst, const float *weights, uint64_t n_edges,
                           uint64_t n, int symmetrise, int64_t *indptr, uint32_t *indices, float *out_weights,
                           uint64_t capacity, uint64_t *nnz_out, std::string &error,
                           ResidentCsr *resident = nullptr);
cudaError_t synthetic_csr(int kind, uint64_t n, uint32_t scale, uint64_t m, uint64_t seed,
                          unsigned long long t_a, unsigned long long t_ab, unsigned long long t_abc,
                          int64_t *indptr, uint32_t *indices, uint64_t capacity, uint64_t *nnz_out,
                          std::string &error, ResidentCsr *resident = nullptr);

}  // namespace b2e

struct b2e_graph {
    b2e::ResidentCsr csr;
    int device = 0;
    int references = 1;  // the caller's object + every handle that walks on it
};

namespace b2e {

// drops one reference; the last one frees the CSR
inline void release_graph(b2e_graph *g) {
    if (g && --g->references == 0) delete g;
}
struct GraphRelease {
    void operator()(b2e_graph *g) const { release_graph(g); }
};

// what a handle holds for its current graph, dropped as a whole when the graph goes
struct HandleGraph {
    std::unique_ptr<b2e_graph, GraphRelease> csr;  // one reference to the graph the handle walks on
    DeviceBuffer<uint2> edge_alias;
    DeviceBuffer<uint32_t> node_types, edge_types;
    GloveState glove;
    DeviceBuffer<uint32_t> walk_raw;  // Walklets: the chunk as walked, before it is split by stride
    DeviceBuffer<uint32_t> sources;
    DeviceBuffer<unsigned long long> filter;  // row filters of the adjacency check (second-order walks)
    DeviceBuffer<uint2> alias;
    DeviceBuffer<float> t0, t1;
    DeviceBuffer<uint32_t> walks[2];
};

}  // namespace b2e

struct b2e_handle {
    b2e_config cfg;
    b2e::HandleGraph graph;
    int sm_count = 0;
    uint64_t n = 0, nnz = 0, n_src = 0;
    uint32_t row_stride = 0;
    uint32_t max_degree = 0;
    uint64_t fold_excess = 0;                // see WalkParams
    unsigned long long thr_fold[3] = {0, 0, 0};
    uint64_t chunk_cap = 0;
    uint64_t slot_first[2] = {0, 0}, slot_count[2] = {0, 0}, slot_stride[2] = {1, 1};
    cudaEvent_t walk_done[2] = {nullptr, nullptr}, train_done[2] = {nullptr, nullptr};
    cudaStream_t walk_stream = nullptr, train_stream = nullptr;
    bool own_streams = false;
    b2e::DeviceBuffer<b2e::DeviceCounters> d_counters;
    unsigned long long thr[3] = {0, 0, 0};
    bool second_order = false;
    bool undirected = false;
    uint64_t launches = 0;
    std::vector<uint32_t> h_alias_thr, h_alias_idx;
    // the exchange step: replicas of the tables on the other GPUs of the node
    uint32_t world = 1, rank = 0;
    float *peer_t0[B2E_MAX_WORLD] = {nullptr}, *peer_t1[B2E_MAX_WORLD] = {nullptr};
    bool peers_are_ipc = false;
};
