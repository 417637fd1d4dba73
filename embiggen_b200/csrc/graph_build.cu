// Graph ingest on the GPU (SURVEY.md 8(f) row 1): edge list -> sorted, de-duplicated,
// self-loop-free CSR, and the seeded synthetic generators of the BASELINE.json shapes.
//
// The reference receives a ready `ensmallen.Graph`; the only in-tree idiom for building one is
// the GraphBuilder loop of /root/reference/embiggen/utils/networkx_utils.py:79-113, and the CSR
// it hands over is described at .../embedders/pecanpy_embedders/node2vec.py:139-163 (rows
// sorted ascending).  This file produces exactly that layout.  Sorting / compaction are
// library calls (CUB ships with the CUDA toolkit); this is the step before the hot path, not
// the hot path.
//
// Synthetic graphs are "the first m distinct undirected edges, in draw order, of the Philox
// stream (seed, draw index)" -- the same definition embiggen_b200/graph.py implements in
// numpy, so both produce the same graph (tests/test_gpu_graph_build.py).
#include <cub/cub.cuh>

#include <algorithm>
#include <string>

#include "host.cuh"

namespace b2e {

constexpr uint32_t TAG_ER = 0x10u;    // graph.py: erdos_renyi
constexpr uint32_t TAG_RMAT = 0x11u;  // graph.py: rmat
constexpr unsigned long long INVALID_KEY = ~0ull;

// candidate undirected edge of draw `idx`: key = (min << 32) | max, INVALID_KEY if rejected
__global__ void __launch_bounds__(256) draw_edges_kernel(int kind, uint64_t n, uint32_t scale,
                                                         uint32_t seed_lo, uint32_t seed_hi,
                                                         unsigned long long t_a, unsigned long long t_ab,
                                                         unsigned long long t_abc, uint64_t first_idx,
                                                         uint64_t count, unsigned long long *keys,
                                                         unsigned long long *ids) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const uint64_t idx = first_idx + k;
    const uint32_t lo = (uint32_t)idx, hi = (uint32_t)(idx >> 32);
    uint64_t u = 0, v = 0;
    if (kind == 0) {
        const uint4 r = philox4x32_10(seed_lo, seed_hi, lo, hi, 0u, TAG_ER << 24);
        u = __umulhi(r.x, (uint32_t)n);
        v = __umulhi(r.y, (uint32_t)n);
    } else {
        for (uint32_t block = 0; block * 4u < scale; ++block) {
            const uint4 r = philox4x32_10(seed_lo, seed_hi, lo, hi, block, TAG_RMAT << 24);
            const uint32_t words[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (uint32_t level = 0; level < 4u; ++level) {
                if (block * 4u + level >= scale) break;
                const unsigned long long w = words[level];
                const uint64_t bit_u = w >= t_ab;
                const uint64_t bit_v = ((w >= t_a) && (w < t_ab)) || (w >= t_abc);
                u = (u << 1) | bit_u;
                v = (v << 1) | bit_v;
            }
        }
    }
    const bool ok = u != v && u < n && v < n;
    const uint64_t a = u < v ? u : v, b = u < v ? v : u;
    keys[k] = ok ? ((a << 32) | b) : INVALID_KEY;
    ids[k] = idx;
}

// (src, dst) host-style edge list -> directed keys (src << 32) | dst, self-loops dropped; originals
// at [0, count), mirrors at [count, 2 count).  With `weights` every key carries its edge's weight in
// `values` (same layout), and flags |= 2 marks a negative or NaN input weight (flags |= 1: an
// endpoint out of range)
__global__ void __launch_bounds__(256) edge_keys_kernel(const uint32_t *src, const uint32_t *dst,
                                                        const float *weights, uint64_t count, uint64_t n,
                                                        int symmetrise, unsigned long long *keys,
                                                        float *values, int *flags) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const uint64_t s = src[k], d = dst[k];
    if (s >= n || d >= n) atomicOr(flags, 1);
    const bool ok = s != d && s < n && d < n;
    keys[k] = ok ? ((s << 32) | d) : INVALID_KEY;
    if (symmetrise) keys[count + k] = ok ? ((d << 32) | s) : INVALID_KEY;
    if (weights) {
        const float w = weights[k];
        if (!(w >= 0.0f)) atomicOr(flags, 2);
        values[k] = w;
        if (symmetrise) values[count + k] = w;
    }
}

__global__ void __launch_bounds__(256) mirror_keys_kernel(const unsigned long long *undirected,
                                                          uint64_t count, unsigned long long *directed) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const unsigned long long key = undirected[k];
    directed[k] = key;
    directed[count + k] = (key << 32) | (key >> 32);
}

// sorted unique directed keys -> indices (low word) and indptr (lower bound of every row start)
__global__ void __launch_bounds__(256) csr_from_keys_kernel(const unsigned long long *keys, uint64_t nnz,
                                                            uint64_t n, uint32_t *indices,
                                                            long long *indptr) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < nnz) indices[k] = (uint32_t)keys[k];
    if (k <= n) {
        const unsigned long long target = (unsigned long long)k << 32;
        uint64_t lo = 0, hi = nnz;
        while (lo < hi) {
            const uint64_t mid = lo + ((hi - lo) >> 1);
            if (keys[mid] < target) lo = mid + 1; else hi = mid;
        }
        indptr[k] = (long long)lo;
    }
}

static inline unsigned blocks_for(uint64_t count) { return (unsigned)((count + 255) / 256); }

// stable radix sort of (keys, values) by key; results land in keys_out / values_out
static cudaError_t sort_pairs(DeviceBuffer<> &temp, const unsigned long long *keys_in,
                              unsigned long long *keys_out, const unsigned long long *values_in,
                              unsigned long long *values_out, uint64_t count, std::string &error) {
    size_t bytes = 0;
    CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys_in, keys_out, values_in, values_out, count));
    CUDA_CHECK(temp.reserve(bytes));
    CUDA_CHECK(cub::DeviceRadixSort::SortPairs(temp.get(), bytes, keys_in, keys_out, values_in, values_out, count));
    return cudaSuccess;
}

static cudaError_t sort_keys(DeviceBuffer<> &temp, const unsigned long long *keys_in,
                             unsigned long long *keys_out, uint64_t count, std::string &error) {
    size_t bytes = 0;
    CUDA_CHECK(cub::DeviceRadixSort::SortKeys(nullptr, bytes, keys_in, keys_out, count));
    CUDA_CHECK(temp.reserve(bytes));
    CUDA_CHECK(cub::DeviceRadixSort::SortKeys(temp.get(), bytes, keys_in, keys_out, count));
    return cudaSuccess;
}

// directed keys (any order) -> CSR in device buffers.  `scratch` is the alternate buffer of the
// radix sort (no third copy).  With `dedup` the keys may repeat and contain INVALID_KEY.  With
// `values` (and their alternate `value_scratch`) every key carries a weight: the sort is stable,
// so the first element of a run of equal keys carries the weight of the key's first occurrence,
// and that is the weight the de-duplicated edge keeps (d_weights, nnz entries).
static cudaError_t keys_to_csr(DeviceBuffer<> &temp, unsigned long long *keys, unsigned long long *scratch,
                               uint64_t count, uint64_t n, bool dedup, DeviceBuffer<int64_t> &d_indptr,
                               DeviceBuffer<uint32_t> &d_indices, uint64_t *nnz_out, std::string &error,
                               float *values = nullptr, float *value_scratch = nullptr,
                               DeviceBuffer<float> *d_weights = nullptr) {
    cub::DoubleBuffer<unsigned long long> buffers(keys, scratch);
    cub::DoubleBuffer<float> weights(values, value_scratch);
    size_t bytes = 0;
    if (values) {
        CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, buffers, weights, count));
        CUDA_CHECK(temp.reserve(bytes));
        CUDA_CHECK(cub::DeviceRadixSort::SortPairs(temp.get(), bytes, buffers, weights, count));
    } else {
        CUDA_CHECK(cub::DeviceRadixSort::SortKeys(nullptr, bytes, buffers, count));
        CUDA_CHECK(temp.reserve(bytes));
        CUDA_CHECK(cub::DeviceRadixSort::SortKeys(temp.get(), bytes, buffers, count));
    }
    unsigned long long *sorted = buffers.Current(), *other = buffers.Alternate();
    float *sorted_values = weights.Current();
    uint64_t nnz = count;
    if (dedup) {
        DeviceBuffer<unsigned long long> selected;
        CUDA_CHECK(selected.reserve(sizeof(unsigned long long)));
        if (values) {  // UniqueByKey keeps the first element of every run
            CUDA_CHECK(cub::DeviceSelect::UniqueByKey(nullptr, bytes, sorted, sorted_values, other,
                                                      weights.Alternate(), selected.get(), count));
            CUDA_CHECK(temp.reserve(bytes));
            CUDA_CHECK(cub::DeviceSelect::UniqueByKey(temp.get(), bytes, sorted, sorted_values, other,
                                                      weights.Alternate(), selected.get(), count));
            sorted_values = weights.Alternate();
        } else {
            CUDA_CHECK(cub::DeviceSelect::Unique(nullptr, bytes, sorted, other, selected.get(), count));
            CUDA_CHECK(temp.reserve(bytes));
            CUDA_CHECK(cub::DeviceSelect::Unique(temp.get(), bytes, sorted, other, selected.get(), count));
        }
        unsigned long long unique = 0, last = 0;
        CUDA_CHECK(cudaMemcpy(&unique, selected.get(), sizeof(unique), cudaMemcpyDeviceToHost));
        if (unique) CUDA_CHECK(cudaMemcpy(&last, other + unique - 1, sizeof(last), cudaMemcpyDeviceToHost));
        nnz = unique - ((unique && last == INVALID_KEY) ? 1 : 0);
        sorted = other;
    }
    *nnz_out = nnz;
    CUDA_CHECK(d_indices.reserve(std::max<uint64_t>(nnz, 1) * sizeof(uint32_t)));
    CUDA_CHECK(d_indptr.reserve((n + 1) * sizeof(long long)));
    csr_from_keys_kernel<<<blocks_for(std::max<uint64_t>(nnz, n + 1)), 256>>>(
        sorted, nnz, n, d_indices.get(), reinterpret_cast<long long *>(d_indptr.get()));
    CUDA_CHECK(cudaGetLastError());
    if (values) {
        CUDA_CHECK(d_weights->reserve(std::max<uint64_t>(nnz, 1) * sizeof(float)));
        if (nnz) CUDA_CHECK(cudaMemcpy(d_weights->get(), sorted_values, nnz * sizeof(float), cudaMemcpyDeviceToDevice));
    }
    CUDA_CHECK(cudaDeviceSynchronize());
    return cudaSuccess;
}

// hand the device arrays over: to host buffers, or (out != nullptr) to a resident b2e_graph.
// `d_weights` is empty for an unweighted graph (then `weights` is not touched).
static cudaError_t deliver(DeviceBuffer<int64_t> &d_indptr, DeviceBuffer<uint32_t> &d_indices,
                           DeviceBuffer<float> &d_weights, uint64_t n, uint64_t nnz, int64_t *indptr,
                           uint32_t *indices, float *weights, uint64_t capacity, ResidentCsr *out,
                           std::string &error) {
    if (out) {
        out->indptr = std::move(d_indptr);
        out->indices = std::move(d_indices);
        out->weights = std::move(d_weights);
        out->n = n;
        out->nnz = nnz;
        return cudaSuccess;
    }
    if (nnz > capacity) {
        error = "indices buffer too small for the de-duplicated graph";
        return cudaErrorInvalidValue;
    }
    CUDA_CHECK(cudaMemcpy(indptr, d_indptr.get(), (n + 1) * sizeof(long long), cudaMemcpyDeviceToHost));
    if (nnz) CUDA_CHECK(cudaMemcpy(indices, d_indices.get(), nnz * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (nnz && weights && d_weights.get())
        CUDA_CHECK(cudaMemcpy(weights, d_weights.get(), nnz * sizeof(float), cudaMemcpyDeviceToHost));
    return cudaSuccess;
}

// Peak device memory per input edge, symmetrised: 8 B of endpoints, 32 B of keys (two buffers of
// two directed keys), plus for a weighted list 4 B of input weights and 16 B of sorted values (two
// buffers of two floats); afterwards the CSR (8 B, 8 B more with weights) while the keys still live.
cudaError_t csr_from_edges(const uint32_t *src, const uint32_t *dst, const float *weights, uint64_t n_edges,
                           uint64_t n, int symmetrise, int64_t *indptr, uint32_t *indices, float *out_weights,
                           uint64_t capacity, uint64_t *nnz_out, std::string &error, ResidentCsr *resident) {
    const uint64_t count = n_edges * (symmetrise ? 2 : 1);
    DeviceBuffer<uint32_t> d_src, d_dst;
    DeviceBuffer<float> d_in, values, value_scratch;
    DeviceBuffer<unsigned long long> keys, scratch;
    DeviceBuffer<> temp;
    DeviceBuffer<int> flag;
    CUDA_CHECK(d_src.reserve(std::max<uint64_t>(n_edges, 1) * sizeof(uint32_t)));
    CUDA_CHECK(d_dst.reserve(std::max<uint64_t>(n_edges, 1) * sizeof(uint32_t)));
    CUDA_CHECK(keys.reserve(std::max<uint64_t>(count, 1) * sizeof(unsigned long long)));
    CUDA_CHECK(scratch.reserve(std::max<uint64_t>(count, 1) * sizeof(unsigned long long)));
    if (weights) {
        CUDA_CHECK(d_in.reserve(std::max<uint64_t>(n_edges, 1) * sizeof(float)));
        CUDA_CHECK(values.reserve(std::max<uint64_t>(count, 1) * sizeof(float)));
        CUDA_CHECK(value_scratch.reserve(std::max<uint64_t>(count, 1) * sizeof(float)));
        CUDA_CHECK(cudaMemcpy(d_in.get(), weights, n_edges * sizeof(float), cudaMemcpyHostToDevice));
    }
    CUDA_CHECK(flag.reserve(sizeof(int)));
    CUDA_CHECK(cudaMemset(flag.get(), 0, sizeof(int)));
    CUDA_CHECK(cudaMemcpy(d_src.get(), src, n_edges * sizeof(uint32_t), cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(d_dst.get(), dst, n_edges * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (n_edges) {
        edge_keys_kernel<<<blocks_for(n_edges), 256>>>(d_src.get(), d_dst.get(), d_in.get(), n_edges, n,
                                                       symmetrise, keys.get(), values.get(), flag.get());
        CUDA_CHECK(cudaGetLastError());
    }
    int flags = 0;
    CUDA_CHECK(cudaMemcpy(&flags, flag.get(), sizeof(int), cudaMemcpyDeviceToHost));
    if (flags & 1) {
        error = "an edge endpoint is not below the number of nodes";
        return cudaErrorInvalidValue;
    }
    if (flags & 2) {
        error = "edge weights must be non-negative numbers";
        return cudaErrorInvalidValue;
    }
    d_src.reset();
    d_dst.reset();
    d_in.reset();
    DeviceBuffer<int64_t> d_indptr;
    DeviceBuffer<uint32_t> d_indices;
    DeviceBuffer<float> d_weights;
    CUDA_CHECK(keys_to_csr(temp, keys.get(), scratch.get(), count, n, true, d_indptr, d_indices, nnz_out, error,
                           values.get(), value_scratch.get(), &d_weights));
    return deliver(d_indptr, d_indices, d_weights, n, *nnz_out, indptr, indices, out_weights, capacity, resident,
                   error);
}

// flags[j] = 1 when keys[j] is a real key that the sorted pool does not hold yet
__global__ void __launch_bounds__(256) new_key_flags_kernel(const unsigned long long *keys, uint64_t count,
                                                            const unsigned long long *pool, uint64_t have,
                                                            unsigned char *flags) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const unsigned long long key = keys[k];
    uint64_t lo = 0, hi = have;
    while (lo < hi) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        if (pool[mid] < key) lo = mid + 1; else hi = mid;
    }
    flags[k] = key != INVALID_KEY && !(lo < have && pool[lo] == key);
}

template <typename T>
static cudaError_t select_flagged(DeviceBuffer<> &temp, const T *in, const unsigned char *flags, T *out,
                                  unsigned long long *d_count, uint64_t count, std::string &error) {
    size_t bytes = 0;
    CUDA_CHECK(cub::DeviceSelect::Flagged(nullptr, bytes, in, flags, out, d_count, count));
    CUDA_CHECK(temp.reserve(bytes));
    CUDA_CHECK(cub::DeviceSelect::Flagged(temp.get(), bytes, in, flags, out, d_count, count));
    return cudaSuccess;
}

// The first m distinct undirected edges of the Philox stream, in draw order.  Candidates are
// drawn in batches; a batch is sorted, de-duplicated (earliest draw wins), filtered against the
// sorted pool of edges already kept, and merged into it.  Every pool edge was first drawn before
// any edge of a later batch, so only the last batch can overshoot m, and only its new edges
// need their draw index to be cut back to "the m earliest".  Memory: two pool buffers of m keys
// plus a few batch-sized arrays, which is what makes the 2-billion-edge shape fit one GPU.
cudaError_t synthetic_csr(int kind, uint64_t n, uint32_t scale, uint64_t m, uint64_t seed,
                          unsigned long long t_a, unsigned long long t_ab, unsigned long long t_abc,
                          int64_t *indptr, uint32_t *indices, uint64_t capacity, uint64_t *nnz_out,
                          std::string &error, ResidentCsr *resident) {
    typedef unsigned long long u64;
    const uint64_t batch_max = 1ull << 29;
    DeviceBuffer<u64> pool[2], keys_in, ids_in, keys_sorted, ids_sorted, keys_unique, ids_unique, keys_new,
        ids_new, d_count;
    DeviceBuffer<unsigned char> flags;
    DeviceBuffer<> temp;
    CUDA_CHECK(d_count.reserve(sizeof(u64)));
    CUDA_CHECK(pool[0].reserve(std::max<uint64_t>(m, 1) * sizeof(u64)));
    CUDA_CHECK(pool[1].reserve(std::max<uint64_t>(m, 1) * sizeof(u64)));
    int cur = 0;
    uint64_t have = 0, drawn = 0;
    for (int round = 0; have < m; ++round) {
        if (round > 400) {
            error = "could not draw enough distinct edges (graph too dense for its shape?)";
            return cudaErrorInvalidValue;
        }
        const uint64_t want = std::min<uint64_t>(batch_max, (uint64_t)((double)(m - have) * 1.3) + 1024);
        for (DeviceBuffer<u64> *buffer : {&keys_in, &ids_in, &keys_sorted, &ids_sorted, &keys_unique, &ids_unique,
                                          &keys_new, &ids_new})
            CUDA_CHECK(buffer->reserve(want * sizeof(u64)));
        CUDA_CHECK(flags.reserve(want));
        draw_edges_kernel<<<blocks_for(want), 256>>>(kind, n, scale, (uint32_t)seed, (uint32_t)(seed >> 32),
                                                     t_a, t_ab, t_abc, drawn, want, keys_in.get(),
                                                     ids_in.get());
        CUDA_CHECK(cudaGetLastError());
        drawn += want;
        // stable sort by key: equal keys stay in ascending draw order, so "first" = earliest draw
        CUDA_CHECK(sort_pairs(temp, keys_in.get(), keys_sorted.get(), ids_in.get(),
                          ids_sorted.get(), want, error));
        size_t bytes = 0;
        CUDA_CHECK(cub::DeviceSelect::UniqueByKey(nullptr, bytes, keys_sorted.get(), ids_sorted.get(),
                                              keys_unique.get(), ids_unique.get(), d_count.get(),
                                              want));
        CUDA_CHECK(temp.reserve(bytes));
        CUDA_CHECK(cub::DeviceSelect::UniqueByKey(temp.get(), bytes, keys_sorted.get(), ids_sorted.get(),
                                              keys_unique.get(), ids_unique.get(), d_count.get(),
                                              want));
        u64 unique = 0;
        CUDA_CHECK(cudaMemcpy(&unique, d_count.get(), sizeof(unique), cudaMemcpyDeviceToHost));
        if (unique == 0) continue;
        new_key_flags_kernel<<<blocks_for(unique), 256>>>(keys_unique.get(), unique, pool[cur].get(),
                                                          have, flags.get());
        CUDA_CHECK(cudaGetLastError());
        CUDA_CHECK(select_flagged(temp, keys_unique.get(), flags.get(), keys_new.get(),
                              d_count.get(), unique, error));
        CUDA_CHECK(select_flagged(temp, ids_unique.get(), flags.get(), ids_new.get(),
                              d_count.get(), unique, error));
        u64 fresh = 0;
        CUDA_CHECK(cudaMemcpy(&fresh, d_count.get(), sizeof(fresh), cudaMemcpyDeviceToHost));
        if (fresh == 0) continue;
        if (have + fresh > m) {  // the last batch overshoots: keep its m - have earliest draws
            const uint64_t keep = m - have;
            CUDA_CHECK(sort_pairs(temp, ids_new.get(), ids_sorted.get(), keys_new.get(),
                              keys_sorted.get(), fresh, error));
            CUDA_CHECK(sort_keys(temp, keys_sorted.get(), keys_new.get(), keep, error));
            fresh = keep;
        }
        CUDA_CHECK(cub::DeviceMerge::MergeKeys(nullptr, bytes, pool[cur].get(), (int64_t)have,
                                           keys_new.get(), (int64_t)fresh, pool[cur ^ 1].get()));
        CUDA_CHECK(temp.reserve(bytes));
        CUDA_CHECK(cub::DeviceMerge::MergeKeys(temp.get(), bytes, pool[cur].get(), (int64_t)have,
                                           keys_new.get(), (int64_t)fresh, pool[cur ^ 1].get()));
        cur ^= 1;
        have += fresh;
    }
    for (DeviceBuffer<u64> *buffer : {&keys_in, &ids_in, &keys_sorted, &ids_sorted, &keys_unique, &ids_unique,
                                      &keys_new, &ids_new})
        buffer->reset();
    flags.reset();
    pool[cur ^ 1].reset();
    // both directions, sorted -> CSR
    DeviceBuffer<u64> directed, alternate;
    CUDA_CHECK(directed.reserve(2 * have * sizeof(u64)));
    mirror_keys_kernel<<<blocks_for(have), 256>>>(pool[cur].get(), have, directed.get());
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaDeviceSynchronize());
    pool[cur].reset();
    CUDA_CHECK(alternate.reserve(2 * have * sizeof(u64)));
    DeviceBuffer<int64_t> d_indptr;
    DeviceBuffer<uint32_t> d_indices;
    DeviceBuffer<float> no_weights;
    CUDA_CHECK(keys_to_csr(temp, directed.get(), alternate.get(), 2 * have, n, false, d_indptr, d_indices,
                       nnz_out, error));
    directed.reset();
    alternate.reset();
    temp.reset();
    return deliver(d_indptr, d_indices, no_weights, n, *nnz_out, indptr, indices, nullptr, capacity, resident,
                   error);
}

}  // namespace b2e
