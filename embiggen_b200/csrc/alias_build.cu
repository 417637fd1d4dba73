// K3 on the GPU: start-node list, maximum degree and the alias table over deg^alpha of the
// negative draws (`use_scale_free_distribution`,
// /root/reference/embiggen/embedders/ensmallen_embedders/node2vec_skipgram.py:101-102), built from
// the device-resident offsets without a pass on the host.
//
// The table is the one oracle/alias.c defines (integer masses m_i, bucket capacity c, light and
// heavy nodes swept in node order), computed in closed form instead of by the sequential sweep.
// With D_k the deficits (c - m) of the light nodes before light node k and S_j the surpluses
// (m - c) of the heavy nodes up to and including heavy node j:
//   light node k  keeps m in its bucket and is topped up by heavy node  #{ j : S_j < D_k };
//   heavy node j  is exhausted by the first light node k with D_k + deficit_k > S_j; it then owns
//                 its bucket with  c + S_j - (D_k + deficit_k)  and is topped up by heavy node
//                 j + 1; a heavy node that is never exhausted owns a full bucket.
// Two compactions, two prefix sums (CUB: library plumbing) and two binary-search kernels; every
// quantity is an integer below 2^62, so the result does not depend on the order of the sums and
// is bit-identical to the oracle's (tests/test_gpu_sgns.py::test_alias_table_bit_exact).
#include <cub/cub.cuh>

#include <cmath>
#include <string>

#include "host.cuh"

namespace b2e {

__device__ __forceinline__ double degree_weight_device(unsigned long long deg, int form) {
    const double d = (double)deg;
    if (deg == 0) return 0.0;
    if (form == 0) return 1.0;                      // alpha = 0
    if (form == 1) return d;                        // alpha = 1
    if (form == 2) return sqrt(d);                  // alpha = 0.5
    return sqrt(sqrt(__dmul_rn(__dmul_rn(d, d), d)));  // alpha = 0.75
}

// offsets sane?  flags |= 4 otherwise (checked before any kernel trusts them)
__global__ void __launch_bounds__(256) indptr_check_kernel(const int64_t *__restrict__ indptr, uint64_t n, uint64_t nnz,
                                                           int *flags) {
    const uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const int64_t a = indptr[v], b = indptr[v + 1];
    if (a < 0 || b < a || (uint64_t)b > nnz) atomicOr(flags, 4);
}

// fixed-point weight of every node (or the host-provided one), "has edges" flag, degree
__global__ void __launch_bounds__(256) alias_weight_kernel(const int64_t *__restrict__ indptr, uint64_t n, int form,
                                                           int bits, const unsigned long long *__restrict__ given,
                                                           unsigned long long *__restrict__ weight,
                                                           uint32_t *__restrict__ has_edges,
                                                           unsigned long long *__restrict__ degree) {
    const uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const unsigned long long deg = (unsigned long long)(indptr[v + 1] - indptr[v]);
    has_edges[v] = deg > 0;
    degree[v] = deg;
    if (weight) weight[v] = given ? given[v] : (unsigned long long)floor(ldexp(degree_weight_device(deg, form), bits));
}

__global__ void __launch_bounds__(256) sources_kernel(const uint32_t *__restrict__ has_edges,
                                                      const uint32_t *__restrict__ rank, uint64_t n,
                                                      uint32_t *__restrict__ sources) {
    const uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n && has_edges[v]) sources[rank[v]] = (uint32_t)v;
}

// final masses and the light flag
__global__ void __launch_bounds__(256) alias_mass_kernel(unsigned long long *__restrict__ mass,
                                                         const uint32_t *__restrict__ has_edges,
                                                         const uint32_t *__restrict__ rank, uint64_t n,
                                                         unsigned long long each, unsigned long long first,
                                                         unsigned long long capacity, uint32_t *__restrict__ is_light) {
    const uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    unsigned long long m = mass[v];
    if (has_edges[v]) m += each + (rank[v] < first ? 1ull : 0ull);
    mass[v] = m;
    is_light[v] = m < capacity;
}

// node ids and deficits / surpluses of the two classes, each in node order
__global__ void __launch_bounds__(256) alias_split_kernel(const unsigned long long *__restrict__ mass,
                                                          const uint32_t *__restrict__ is_light,
                                                          const uint32_t *__restrict__ light_rank, uint64_t n,
                                                          unsigned long long capacity, uint32_t *__restrict__ light,
                                                          uint32_t *__restrict__ heavy,
                                                          unsigned long long *__restrict__ deficit,
                                                          unsigned long long *__restrict__ surplus) {
    const uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const uint32_t k = light_rank[v];
    if (is_light[v]) {
        light[k] = (uint32_t)v;
        deficit[k] = capacity - mass[v];
    } else {
        heavy[v - k] = (uint32_t)v;
        surplus[v - k] = mass[v] - capacity;
    }
}

// floor(mass 2^32 / capacity) for mass < capacity < 2^62 (oracle/alias.c: threshold)
__device__ __forceinline__ uint32_t alias_threshold(unsigned long long mass, unsigned long long capacity) {
    unsigned long long r = mass;
    uint32_t q = 0;
#pragma unroll 4
    for (int bit = 0; bit < 32; ++bit) {
        r <<= 1;
        q <<= 1;
        if (r >= capacity) { r -= capacity; q |= 1u; }
    }
    return q;
}

__global__ void __launch_bounds__(256) alias_light_kernel(const uint32_t *__restrict__ light,
                                                          const uint32_t *__restrict__ heavy,
                                                          const unsigned long long *__restrict__ deficit,
                                                          const unsigned long long *__restrict__ deficit_sum,
                                                          const unsigned long long *__restrict__ surplus_sum,
                                                          uint64_t n_light, uint64_t n_heavy,
                                                          unsigned long long capacity, uint2 *__restrict__ table) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_light) return;
    const unsigned long long before = deficit_sum[k] - deficit[k];
    uint64_t lo = 0, hi = n_heavy;  // heavy nodes exhausted before this one: surplus_sum < before
    while (lo < hi) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(surplus_sum + mid) < before) lo = mid + 1; else hi = mid;
    }
    table[light[k]] = make_uint2(alias_threshold(capacity - deficit[k], capacity), heavy[lo]);
}

__global__ void __launch_bounds__(256) alias_heavy_kernel(const uint32_t *__restrict__ heavy,
                                                          const unsigned long long *__restrict__ deficit_sum,
                                                          const unsigned long long *__restrict__ surplus_sum,
                                                          uint64_t n_light, uint64_t n_heavy,
                                                          unsigned long long capacity, uint2 *__restrict__ table) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_heavy) return;
    const unsigned long long mine = surplus_sum[j];
    uint64_t lo = 0, hi = n_light;  // first light node whose running deficit exceeds my running surplus
    while (lo < hi) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(deficit_sum + mid) > mine) hi = mid; else lo = mid + 1;
    }
    const uint32_t v = heavy[j];
    if (lo >= n_light || j + 1 >= n_heavy) {
        table[v] = make_uint2(0xFFFFFFFFu, v);  // never exhausted: a full bucket
    } else {
        table[v] = make_uint2(alias_threshold(capacity + mine - deficit_sum[lo], capacity), heavy[j + 1]);
    }
}

static inline unsigned grid_for(uint64_t count) { return (unsigned)((count + 255) / 256); }

static int exact_form(double alpha) {
    if (alpha == 0.0) return 0;
    if (alpha == 1.0) return 1;
    if (alpha == 0.5) return 2;
    if (alpha == 0.75) return 3;
    return -1;
}

static double degree_weight_host(uint64_t deg, double alpha) {
    const double d = (double)deg;
    if (deg == 0) return 0.0;
    if (alpha == 0.0) return 1.0;
    if (alpha == 1.0) return d;
    if (alpha == 0.5) return std::sqrt(d);
    if (alpha == 0.75) return std::sqrt(std::sqrt(d * d * d));
    return std::pow(d, alpha);
}

int alias_fraction_bits(uint64_t n, uint64_t max_degree, double alpha) {
    const double w_max = degree_weight_host(max_degree, alpha);
    int bits = 40;
    while (bits > 0 && (double)n * (std::floor(std::ldexp(w_max, bits)) + 1.0) >= 4611686018427387904.0) --bits;
    return bits;
}

cudaError_t check_indptr_device(const int64_t *d_indptr, uint64_t n, uint64_t nnz, int *d_flags, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    indptr_check_kernel<<<grid_for(n), 256, 0, stream>>>(d_indptr, n, nnz, d_flags);
    return cudaGetLastError();
}

// Start nodes (always) and the alias table (when `d_table` is given) from the device offsets.
// `host_indptr` is needed only for an exponent without an exact form (libm's pow is the oracle's).
cudaError_t build_node_tables(const int64_t *d_indptr, const int64_t *host_indptr, uint64_t n, double alpha,
                              uint32_t *d_sources, uint64_t *n_src_out, uint64_t *max_degree_out, uint2 *d_table,
                              cudaStream_t stream, std::string &error) {
    typedef unsigned long long u64;
    DeviceBuffer<u64> weight, degree, scalar, given;
    DeviceBuffer<uint32_t> has_edges, rank;
    DeviceBuffer<> temp;
    CUDA_CHECK(has_edges.reserve(n * sizeof(uint32_t)));
    CUDA_CHECK(rank.reserve(n * sizeof(uint32_t)));
    CUDA_CHECK(degree.reserve(n * sizeof(u64)));
    CUDA_CHECK(scalar.reserve(2 * sizeof(u64)));
    size_t bytes = 0, need = 0;
    // pass 1: degrees, flags; the largest degree fixes the fixed-point format
    alias_weight_kernel<<<grid_for(n), 256, 0, stream>>>(d_indptr, n, 0, 0, nullptr, nullptr, has_edges.get(),
                                                         degree.get());
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cub::DeviceReduce::Max(nullptr, bytes, degree.get(), scalar.get(), n, stream));
    need = bytes;
    CUDA_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, bytes, has_edges.get(), rank.get(), n, stream));
    need = std::max(need, bytes);
    CUDA_CHECK(cub::DeviceScan::InclusiveSum(nullptr, bytes, degree.get(), degree.get(), n, stream));
    need = std::max(need, bytes);
    CUDA_CHECK(cub::DeviceReduce::Sum(nullptr, bytes, degree.get(), scalar.get(), n, stream));
    need = std::max(need, bytes);
    CUDA_CHECK(temp.reserve(std::max<size_t>(need, 1)));
    bytes = need;
    CUDA_CHECK(cub::DeviceReduce::Max(temp.get(), bytes, degree.get(), scalar.get(), n, stream));
    bytes = need;
    CUDA_CHECK(cub::DeviceScan::ExclusiveSum(temp.get(), bytes, has_edges.get(), rank.get(), n, stream));
    sources_kernel<<<grid_for(n), 256, 0, stream>>>(has_edges.get(), rank.get(), n, d_sources);
    CUDA_CHECK(cudaGetLastError());
    u64 max_degree = 0;
    uint32_t last_rank = 0, last_flag = 0;
    CUDA_CHECK(cudaMemcpyAsync(&max_degree, scalar.get(), sizeof(u64), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaMemcpyAsync(&last_rank, rank.get() + (n - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaMemcpyAsync(&last_flag, has_edges.get() + (n - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    const uint64_t n_src = (uint64_t)last_rank + last_flag;
    *n_src_out = n_src;
    *max_degree_out = max_degree;
    if (!d_table) return cudaSuccess;
    if (n_src == 0) {
        error = "alias table: total weight is zero";
        return cudaErrorInvalidValue;
    }

    // pass 2: fixed-point weights and their total
    const int bits = alias_fraction_bits(n, max_degree, alpha);
    const int form = exact_form(alpha);
    CUDA_CHECK(weight.reserve(n * sizeof(u64)));
    if (form < 0) {  // libm's pow on the host, like the oracle; one upload of 8 bytes per node
        if (!host_indptr) {
            error = "a negative_sampling_exponent other than 0, 0.5, 0.75, 1 needs the offsets on the host";
            return cudaErrorInvalidValue;
        }
        std::vector<u64> host(n);
        for (uint64_t v = 0; v < n; ++v)
            host[v] = (u64)std::floor(std::ldexp(degree_weight_host((uint64_t)(host_indptr[v + 1] - host_indptr[v]), alpha), bits));
        CUDA_CHECK(given.reserve(n * sizeof(u64)));
        CUDA_CHECK(cudaMemcpyAsync(given.get(), host.data(), n * sizeof(u64), cudaMemcpyHostToDevice, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
    }
    alias_weight_kernel<<<grid_for(n), 256, 0, stream>>>(d_indptr, n, form < 0 ? 0 : form, bits,
                                                         form < 0 ? given.get() : nullptr, weight.get(),
                                                         has_edges.get(), degree.get());
    CUDA_CHECK(cudaGetLastError());
    bytes = need;
    CUDA_CHECK(cub::DeviceReduce::Sum(temp.get(), bytes, weight.get(), scalar.get(), n, stream));
    u64 total = 0;
    CUDA_CHECK(cudaMemcpyAsync(&total, scalar.get(), sizeof(u64), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    if (total == 0) {
        error = "alias table: total weight is zero";
        return cudaErrorInvalidValue;
    }
    const u64 capacity = (total + n - 1) / n;
    const u64 excess = capacity * n - total, each = excess / n_src, first = excess % n_src;

    // pass 3: masses, classes, the two node lists with their deficits / surpluses
    DeviceBuffer<uint32_t> is_light, light_rank, light, heavy;
    DeviceBuffer<u64> deficit, surplus;
    CUDA_CHECK(is_light.reserve(n * sizeof(uint32_t)));
    CUDA_CHECK(light_rank.reserve(n * sizeof(uint32_t)));
    alias_mass_kernel<<<grid_for(n), 256, 0, stream>>>(weight.get(), has_edges.get(), rank.get(), n,
                                                       each, first, capacity, is_light.get());
    CUDA_CHECK(cudaGetLastError());
    bytes = need;
    CUDA_CHECK(cub::DeviceScan::ExclusiveSum(temp.get(), bytes, is_light.get(), light_rank.get(), n, stream));
    uint32_t tail_rank = 0, tail_flag = 0;
    CUDA_CHECK(cudaMemcpyAsync(&tail_rank, light_rank.get() + (n - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaMemcpyAsync(&tail_flag, is_light.get() + (n - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    const uint64_t n_light = (uint64_t)tail_rank + tail_flag, n_heavy = n - n_light;
    if (n_heavy == 0) {  // impossible: the masses add up to n capacities
        error = "alias table: no heavy node";
        return cudaErrorInvalidValue;
    }
    CUDA_CHECK(light.reserve(std::max<size_t>(n_light * sizeof(uint32_t), 1)));
    CUDA_CHECK(heavy.reserve(n_heavy * sizeof(uint32_t)));
    CUDA_CHECK(deficit.reserve(std::max<size_t>(n_light * sizeof(u64), 1)));
    CUDA_CHECK(surplus.reserve(n_heavy * sizeof(u64)));
    alias_split_kernel<<<grid_for(n), 256, 0, stream>>>(weight.get(), is_light.get(),
                                                        light_rank.get(), n, capacity, light.get(),
                                                        heavy.get(), deficit.get(), surplus.get());
    CUDA_CHECK(cudaGetLastError());
    // running sums: the deficits keep their own copy (the light kernel needs both), in `degree`
    u64 *deficit_sum = degree.get();
    if (n_light) {
        bytes = need;
        CUDA_CHECK(cub::DeviceScan::InclusiveSum(temp.get(), bytes, deficit.get(), deficit_sum, n_light, stream));
    }
    bytes = need;
    CUDA_CHECK(cub::DeviceScan::InclusiveSum(temp.get(), bytes, surplus.get(), surplus.get(), n_heavy, stream));
    if (n_light) {
        alias_light_kernel<<<grid_for(n_light), 256, 0, stream>>>(light.get(), heavy.get(),
                                                                  deficit.get(), deficit_sum, surplus.get(),
                                                                  n_light, n_heavy, capacity, d_table);
        CUDA_CHECK(cudaGetLastError());
    }
    alias_heavy_kernel<<<grid_for(n_heavy), 256, 0, stream>>>(heavy.get(), deficit_sum, surplus.get(), n_light,
                                                              n_heavy, capacity, d_table);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaStreamSynchronize(stream));
    return cudaSuccess;
}


// ---- per-row alias tables of a weighted graph (the proposal of weighted walks) ----
// The normative construction is oracle/walks.c: orc_edge_alias, reproduced bit for bit: per row of
// d edges, total = the left-to-right double sum of its weights, heaviest = the first index of the
// strict maximum, scaled_i = w_i d / total (1 when total is 0), small / large = LIFO stacks filled
// in ascending edge order, thr = min(floor(scaled 2^32), 2^32 - 1), leftovers {2^32 - 1, self}
// except a zero-weight leftover, {0, heaviest}.  The double operations are the _rn intrinsics so
// that nothing is contracted into an FMA.  LIFO Vose is sequential within a row, so one thread
// builds one row; the threads take the rows longest first (the longest row is the critical path).
// Each row keeps its open scaled_i in its own 8-byte output slot, which becomes {thr, alias} when
// entry i closes, and both stacks in one two-ended array of 4 B per edge at the row's offset:
// small grows up from the front, large down from the back (|small| + |large| <= d).

__global__ void __launch_bounds__(256) row_degree_kernel(const int64_t *__restrict__ indptr, uint64_t n,
                                                         uint32_t *__restrict__ degree, uint32_t *__restrict__ row) {
    const uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    degree[v] = (uint32_t)(indptr[v + 1] - indptr[v]);
    row[v] = (uint32_t)v;
}

// a table slot: low word thr, high word alias (the layout of uint2 {x = thr, y = alias})
__device__ __forceinline__ unsigned long long edge_entry(uint32_t thr, uint32_t alias) {
    return ((unsigned long long)alias << 32) | thr;
}

__global__ void __launch_bounds__(128) edge_alias_kernel(const int64_t *__restrict__ indptr,
                                                         const uint32_t *__restrict__ order, uint64_t n,
                                                         const float *__restrict__ weights,
                                                         unsigned long long *__restrict__ table,
                                                         uint32_t *__restrict__ stacks, int *flags) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint32_t v = order[t];
    const int64_t begin = indptr[v];
    const uint64_t d = (uint64_t)(indptr[v + 1] - begin);
    if (d == 0) return;
    const float *w = weights + begin;
    unsigned long long *slot = table + begin;
    uint32_t *stack = stacks + begin;
    double total = 0.0;
    uint64_t heaviest = 0;
    float w_heaviest = w[0];
    for (uint64_t i = 0; i < d; ++i) {
        const float wi = w[i];
        if (!(wi >= 0.0f)) {  // negative or NaN
            atomicOr(flags, 1);
            return;
        }
        total = __dadd_rn(total, (double)wi);
        if (wi > w_heaviest) {
            heaviest = i;
            w_heaviest = wi;
        }
    }
    const double dd = (double)d;
    uint64_t ns = 0, nl = 0;  // small: stack[0, ns); large: stack[d - nl, d), top at stack[d - nl]
    for (uint64_t i = 0; i < d; ++i) {
        const double scaled = total > 0.0 ? __ddiv_rn(__dmul_rn((double)w[i], dd), total) : 1.0;
        slot[i] = (unsigned long long)__double_as_longlong(scaled);
        if (scaled < 1.0) stack[ns++] = (uint32_t)i; else stack[d - 1 - nl++] = (uint32_t)i;
    }
    while (ns > 0 && nl > 0) {
        const uint32_t s = stack[--ns];
        const uint32_t l = stack[d - nl];
        --nl;
        const double scaled_s = __longlong_as_double((long long)slot[s]);
        const double thr = floor(__dmul_rn(scaled_s, 4294967296.0));
        slot[s] = edge_entry(thr >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)thr, l);
        const double scaled_l = __dsub_rn(__dadd_rn(__longlong_as_double((long long)slot[l]), scaled_s), 1.0);
        slot[l] = (unsigned long long)__double_as_longlong(scaled_l);
        if (scaled_l < 1.0) stack[ns++] = l; else stack[d - 1 - nl++] = l;
    }
    for (uint64_t k = 0; k < ns; ++k) {  // leftovers of weight zero are never proposed
        const uint32_t s = stack[k];
        slot[s] = total > 0.0 && w[s] == 0.0f ? edge_entry(0u, (uint32_t)heaviest) : edge_entry(0xFFFFFFFFu, s);
    }
    for (uint64_t k = 0; k < nl; ++k) {
        const uint32_t l = stack[d - 1 - k];
        slot[l] = edge_entry(0xFFFFFFFFu, l);
    }
}

// normalize_by_degree (oracle: degree_normalised_weights): one IEEE float division per edge
__global__ void __launch_bounds__(256) degree_normalise_kernel(const int64_t *__restrict__ indptr,
                                                               const uint32_t *__restrict__ indices,
                                                               const float *__restrict__ weights, uint64_t nnz,
                                                               float *__restrict__ out) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    const uint32_t x = indices[e];
    const long long degree = (long long)(indptr[x + 1] - indptr[x]);
    out[e] = __fdiv_rn(weights ? weights[e] : 1.0f, (float)(degree > 1 ? degree : 1));
}

cudaError_t launch_degree_normalise(const int64_t *d_indptr, const uint32_t *d_indices, const float *d_weights,
                                    uint64_t nnz, float *d_out, cudaStream_t stream) {
    if (nnz == 0) return cudaSuccess;
    degree_normalise_kernel<<<grid_for(nnz), 256, 0, stream>>>(d_indptr, d_indices, d_weights, nnz, d_out);
    return cudaGetLastError();
}

// Device memory beyond the table (8 B per edge): 4 B per edge of stacks and 16 B per node for the
// degree-sorted row order.
cudaError_t build_edge_alias(const int64_t *d_indptr, const float *d_weights, uint64_t n, uint64_t nnz,
                             uint2 *d_table, uint64_t *longest_row, cudaStream_t stream, std::string &error) {
    DeviceBuffer<uint32_t> degree, degree_sorted, row, order, stacks;
    DeviceBuffer<int> flags;
    DeviceBuffer<> temp;
    CUDA_CHECK(degree.reserve(n * sizeof(uint32_t)));
    CUDA_CHECK(degree_sorted.reserve(n * sizeof(uint32_t)));
    CUDA_CHECK(row.reserve(n * sizeof(uint32_t)));
    CUDA_CHECK(order.reserve(n * sizeof(uint32_t)));
    CUDA_CHECK(stacks.reserve(std::max<uint64_t>(nnz, 1) * sizeof(uint32_t)));
    CUDA_CHECK(flags.reserve(sizeof(int)));
    CUDA_CHECK(cudaMemsetAsync(flags.get(), 0, sizeof(int), stream));
    row_degree_kernel<<<grid_for(n), 256, 0, stream>>>(d_indptr, n, degree.get(), row.get());
    CUDA_CHECK(cudaGetLastError());
    size_t bytes = 0;
    CUDA_CHECK(cub::DeviceRadixSort::SortPairsDescending(nullptr, bytes, degree.get(), degree_sorted.get(), row.get(),
                                                         order.get(), n, 0, 32, stream));
    CUDA_CHECK(temp.reserve(std::max<size_t>(bytes, 1)));
    CUDA_CHECK(cub::DeviceRadixSort::SortPairsDescending(temp.get(), bytes, degree.get(), degree_sorted.get(),
                                                         row.get(), order.get(), n, 0, 32, stream));
    edge_alias_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(
        d_indptr, order.get(), n, d_weights, reinterpret_cast<unsigned long long *>(d_table), stacks.get(),
        flags.get());
    CUDA_CHECK(cudaGetLastError());
    int bad = 0;
    uint32_t longest = 0;
    CUDA_CHECK(cudaMemcpyAsync(&bad, flags.get(), sizeof(int), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaMemcpyAsync(&longest, degree_sorted.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    if (bad) {
        error = "edge weights must be non-negative numbers";
        return cudaErrorInvalidValue;
    }
    *longest_row = longest;
    return cudaSuccess;
}

}  // namespace b2e
