// The one exchange step of the path (SURVEY.md 8e): data-parallel replicas of the two embedding
// tables, one per GPU, are averaged at a fixed step interval.  The reference has no counterpart
// (one shared table in host RAM, /root/reference/embiggen/embedders/ensmallen_embedders/node2vec.py:99
// runs on one machine's cores); north_star prescribes the averaging.
//
// Instead of handing the padded tables to a library all-reduce, one kernel does the reduction
// and the redistribution over NVLink / NVSwitch peer memory: rank r owns the rows
// [n r / G, n (r + 1) / G); a warp gathers the G replicas of an owned row with peer loads (only
// the ceil(D / 4) chunks that hold data travel -- the 128 B row padding never crosses a link),
// sums them in rank order, scales by 1 / G and scatters the result to all G replicas with peer
// stores.  Per GPU and direction (G - 1) / G of the live table bytes cross NVLink once; nothing
// is staged, nothing is packed.  The sum order is fixed, so the replicas are bit-identical
// afterwards.  Peers are opened through CUDA IPC (one process per GPU) or passed directly
// (several handles in one process: tests).  The caller brackets the kernel with a barrier on both
// sides (every replica finished its SGD chunk; every owner finished writing).
#include <algorithm>

#include "common.cuh"

namespace b2e {

struct ExchangeParams {
    float *t[2][B2E_MAX_WORLD];
    uint32_t world;
    uint64_t row_begin, row_end;
    uint32_t row_stride, chunks;
    float scale;
};

// One warp per (table, row), U rows per iteration: the G x U loads of a lane are issued back to
// back before the first is consumed.  Measured at G = 2 on C5 (80 GB per direction and exchange):
// 125 ms for U = 1, 4 and 8 alike (profiles/r02m_*): 637 GB/s per direction, bound by the links.
template <int G, int U>
__global__ void __launch_bounds__(256) exchange_average_kernel(const ExchangeParams p) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t rows = p.row_end - p.row_begin, items = 2 * rows;
    constexpr int GG = G ? G : B2E_MAX_WORLD;
    const uint32_t world = G ? (uint32_t)G : p.world;
    for (uint64_t base = (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * U; base < items;
         base += warps * U) {
        for (uint32_t c = lane; c < p.chunks; c += 32u) {
            float4 v[U][GG];
            uint64_t at[U];
            uint32_t table[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint64_t item = base + u < items ? base + u : items - 1;  // the tail repeats its last row
                table[u] = item >= rows;
                at[u] = (p.row_begin + (table[u] ? item - rows : item)) * p.row_stride;
#pragma unroll
                for (int g = 0; g < GG; ++g)
                    if ((uint32_t)g < world) v[u][g] = __ldcg(reinterpret_cast<const float4 *>(p.t[table[u]][g] + at[u]) + c);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                float4 s = v[u][0];
#pragma unroll
                for (int g = 1; g < GG; ++g) {
                    if ((uint32_t)g < world) {
                        s.x = __fadd_rn(s.x, v[u][g].x);
                        s.y = __fadd_rn(s.y, v[u][g].y);
                        s.z = __fadd_rn(s.z, v[u][g].z);
                        s.w = __fadd_rn(s.w, v[u][g].w);
                    }
                }
                s.x = __fmul_rn(s.x, p.scale);
                s.y = __fmul_rn(s.y, p.scale);
                s.z = __fmul_rn(s.z, p.scale);
                s.w = __fmul_rn(s.w, p.scale);
                if (base + u < items) {
#pragma unroll
                    for (int g = 0; g < GG; ++g)
                        if ((uint32_t)g < world) __stcg(reinterpret_cast<float4 *>(p.t[table[u]][g] + at[u]) + c, s);
                }
            }
        }
    }
}

cudaError_t launch_exchange_average(float *const t0[], float *const t1[], uint32_t world, uint32_t rank,
                                    uint64_t n, uint32_t row_stride, uint32_t chunks, int sm_count,
                                    cudaStream_t stream) {
    if (world < 2 || n == 0) return cudaSuccess;
    ExchangeParams p;
    for (uint32_t g = 0; g < world; ++g) {
        p.t[0][g] = t0[g];
        p.t[1][g] = t1[g];
    }
    p.world = world;
    p.row_begin = n * rank / world;
    p.row_end = n * (rank + 1ull) / world;
    p.row_stride = row_stride;
    p.chunks = chunks;
    p.scale = 1.0f / (float)world;
    const uint64_t rows = p.row_end - p.row_begin;
    if (rows == 0) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<uint64_t>((2 * rows + 7) / 8, (uint64_t)sm_count * 8);
    // rows per warp iteration: enough loads in flight per lane to cover an NVLink round trip, the
    // G x U loads of a lane held to eight float4
    switch (world) {
        case 2: exchange_average_kernel<2, 4><<<grid, 256, 0, stream>>>(p); break;
        case 4: exchange_average_kernel<4, 2><<<grid, 256, 0, stream>>>(p); break;
        case 8: exchange_average_kernel<8, 1><<<grid, 256, 0, stream>>>(p); break;
        default: exchange_average_kernel<0, 1><<<grid, 256, 0, stream>>>(p); break;
    }
    return cudaGetLastError();
}

// GloVe's merge of a sharded epoch.  Every rank trained only the centres it owns, so averaging the
// replicas would divide each owner's T0 change and each rank's T1 change by G.  Instead: row v of
// T0 is taken from the replica of owner(v) (the only one that changed it), and T1 becomes
// snapshot + ((T1_0 - snapshot) + (T1_1 - snapshot) + ...), rank order, every operation rounded
// to nearest -- the sum of all ranks' changes on the common starting point.  The snapshot is the
// same on every replica (they were bit-identical when it was taken), so each rank reads its own.
// Rows are split among the ranks and moved like exchange_average_kernel's (one warp per (table,
// row), only the ceil(D / 4) live chunks); afterwards the replicas are bit-identical again.
struct GloveMergeParams {
    float *t[2][B2E_MAX_WORLD];
    const float *snapshot;
    uint32_t owner_bounds[B2E_MAX_WORLD + 1];
    uint32_t world;
    uint64_t row_begin, row_end;
    uint32_t row_stride, chunks;
};

template <int G>
__global__ void __launch_bounds__(256) glove_merge_kernel(const GloveMergeParams p) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t rows = p.row_end - p.row_begin, items = 2 * rows;
    constexpr int GG = G ? G : B2E_MAX_WORLD;
    const uint32_t world = G ? (uint32_t)G : p.world;
    for (uint64_t item = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; item < items; item += warps) {
        const bool second = item >= rows;  // warp-uniform
        const uint64_t row = p.row_begin + (second ? item - rows : item), at = row * p.row_stride;
        if (!second) {
            uint32_t owner = 0;  // last rank whose interval starts at or before the row
            while (owner + 1 < world && row >= p.owner_bounds[owner + 1]) ++owner;
            for (uint32_t c = lane; c < p.chunks; c += 32u) {
                const float4 v = __ldcg(reinterpret_cast<const float4 *>(p.t[0][owner] + at) + c);
#pragma unroll
                for (int g = 0; g < GG; ++g)
                    if ((uint32_t)g < world && (uint32_t)g != owner)
                        __stcg(reinterpret_cast<float4 *>(p.t[0][g] + at) + c, v);
            }
            continue;
        }
        for (uint32_t c = lane; c < p.chunks; c += 32u) {
            const float4 s = __ldcg(reinterpret_cast<const float4 *>(p.snapshot + at) + c);
            float4 v[GG];
#pragma unroll
            for (int g = 0; g < GG; ++g)
                if ((uint32_t)g < world) v[g] = __ldcg(reinterpret_cast<const float4 *>(p.t[1][g] + at) + c);
            float4 d = make_float4(__fsub_rn(v[0].x, s.x), __fsub_rn(v[0].y, s.y), __fsub_rn(v[0].z, s.z),
                                   __fsub_rn(v[0].w, s.w));
#pragma unroll
            for (int g = 1; g < GG; ++g) {
                if ((uint32_t)g < world) {
                    d.x = __fadd_rn(d.x, __fsub_rn(v[g].x, s.x));
                    d.y = __fadd_rn(d.y, __fsub_rn(v[g].y, s.y));
                    d.z = __fadd_rn(d.z, __fsub_rn(v[g].z, s.z));
                    d.w = __fadd_rn(d.w, __fsub_rn(v[g].w, s.w));
                }
            }
            const float4 out = make_float4(__fadd_rn(s.x, d.x), __fadd_rn(s.y, d.y), __fadd_rn(s.z, d.z),
                                           __fadd_rn(s.w, d.w));
#pragma unroll
            for (int g = 0; g < GG; ++g)
                if ((uint32_t)g < world) __stcg(reinterpret_cast<float4 *>(p.t[1][g] + at) + c, out);
        }
    }
}

cudaError_t launch_glove_merge(float *const t0[], float *const t1[], const float *snapshot,
                               const uint32_t *owner_bounds, uint32_t world, uint32_t rank, uint64_t n,
                               uint32_t row_stride, uint32_t chunks, int sm_count, cudaStream_t stream) {
    if (world < 2 || n == 0) return cudaSuccess;
    GloveMergeParams p;
    for (uint32_t g = 0; g < world; ++g) {
        p.t[0][g] = t0[g];
        p.t[1][g] = t1[g];
    }
    for (uint32_t r = 0; r <= world; ++r) p.owner_bounds[r] = owner_bounds[r];
    p.snapshot = snapshot;
    p.world = world;
    p.row_begin = n * rank / world;
    p.row_end = n * (rank + 1ull) / world;
    p.row_stride = row_stride;
    p.chunks = chunks;
    const uint64_t rows = p.row_end - p.row_begin;
    if (rows == 0) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<uint64_t>((2 * rows + 7) / 8, (uint64_t)sm_count * 8);
    switch (world) {
        case 2: glove_merge_kernel<2><<<grid, 256, 0, stream>>>(p); break;
        case 4: glove_merge_kernel<4><<<grid, 256, 0, stream>>>(p); break;
        case 8: glove_merge_kernel<8><<<grid, 256, 0, stream>>>(p); break;
        default: glove_merge_kernel<0><<<grid, 256, 0, stream>>>(p); break;
    }
    return cudaGetLastError();
}

// Strip the row padding on the device: `rows` rows of `chunks` float4 each leave their 128 B-aligned
// pitch for a dense buffer that one contiguous DMA then carries to the host (a pitched 2-D copy of
// 400-byte rows moved 80 GB in 12 s; packed and double-buffered it is bound by PCIe).
__global__ void __launch_bounds__(256) pack_rows_kernel(const float *__restrict__ table, uint64_t rows,
                                                        uint32_t row_stride, uint32_t dim, float *__restrict__ dense) {
    const uint64_t total = rows * dim;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total;
         k += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t row = k / dim;
        dense[k] = __ldg(table + row * row_stride + (k - row * dim));
    }
}

cudaError_t launch_pack_rows(const float *table, uint64_t rows, uint32_t row_stride, uint32_t dim, float *dense,
                             int sm_count, cudaStream_t stream) {
    if (rows == 0) return cudaSuccess;
    pack_rows_kernel<<<(unsigned)sm_count * 8u, 256, 0, stream>>>(table, rows, row_stride, dim, dense);
    return cudaGetLastError();
}

// digest of the live part of both tables (replica equality / finiteness checks of the multi-GPU
// path without moving the tables): per table the sum and the sum of squares in double
// (informative: atomics reorder them) and the wrap-around integer sum of the float bit patterns
// (exact and order-independent: equal replicas <=> equal words, up to collisions), then the
// number of non-finite values
struct TablesDigest {
    double sum[2], squares[2];
    unsigned long long bits[2], non_finite;
};

__global__ void __launch_bounds__(256) tables_digest_kernel(const float *__restrict__ t0,
                                                            const float *__restrict__ t1, uint64_t n,
                                                            uint32_t row_stride, uint32_t dim, TablesDigest *out) {
    double sum[2] = {0.0, 0.0}, squares[2] = {0.0, 0.0};
    unsigned long long bits[2] = {0, 0}, bad = 0;
    const uint64_t total = n * dim;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total;
         k += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t row = k / dim, at = row * row_stride + (k - row * dim);
        const float v[2] = {__ldg(t0 + at), __ldg(t1 + at)};
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            if (!isfinite(v[t])) ++bad;
            sum[t] += (double)v[t];
            squares[t] += (double)v[t] * (double)v[t];
            bits[t] += (unsigned long long)__float_as_uint(v[t]) * (2ull * (k % 0x7FFFFFFFull) + 1ull);
        }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            sum[t] += __shfl_xor_sync(0xffffffffu, sum[t], off);
            squares[t] += __shfl_xor_sync(0xffffffffu, squares[t], off);
            bits[t] += __shfl_xor_sync(0xffffffffu, bits[t], off);
        }
        bad += __shfl_xor_sync(0xffffffffu, bad, off);
    }
    if ((threadIdx.x & 31u) == 0) {
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            atomicAdd(&out->sum[t], sum[t]);
            atomicAdd(&out->squares[t], squares[t]);
            atomicAdd(&out->bits[t], bits[t]);
        }
        if (bad) atomicAdd(&out->non_finite, bad);
    }
}

cudaError_t launch_tables_digest(const float *t0, const float *t1, uint64_t n, uint32_t row_stride,
                                 uint32_t dim, void *d_out, int sm_count, cudaStream_t stream) {
    static_assert(sizeof(TablesDigest) == 56, "b2e_tables_digest copies 7 eight-byte words");
    cudaError_t err = cudaMemsetAsync(d_out, 0, sizeof(TablesDigest), stream);
    if (err != cudaSuccess || n == 0) return err;
    tables_digest_kernel<<<(unsigned)sm_count * 8u, 256, 0, stream>>>(t0, t1, n, row_stride, dim,
                                                                      static_cast<TablesDigest *>(d_out));
    return cudaGetLastError();
}

}  // namespace b2e
