// GloVe on random-walk co-occurrences (SURVEY.md 8(f) row 3) for sm_100a.
//
// Counterpart of what `ensmallen.models.GloVe.fit_transform` does behind
// `Node2VecGloVeEnsmallen` / `DeepWalkGloVeEnsmallen`
// (/root/reference/embiggen/embedders/ensmallen_embedders/node2vec_glove.py:5-140,
// deepwalk_glove.py): per epoch one walk per node, the co-occurrence counts of the walks'
// windows, one pass of weighted least squares over the non-zero counts (Pennington et al. 2014,
// eq. 8, no bias terms; normative statement: oracle/glove.c).
//
//   1. cooc_keys_kernel      every (position, offset <= window) of a walk chunk emits the two
//                            ordered keys (centre << 32 | context), or an all-ones key
//   2. CUB radix sort + run-length encode -> (key, count) of the chunk; chunks are merged by
//      sort-by-key + reduce-by-key (library calls: this is bookkeeping around the hot kernel)
//   3. cooc_rowptr_kernel    CSR offsets of the sorted keys by centre (one bisection per node)
//   4. glove_tile_kernel     one warp per tile of 512 consecutive triples (load balance on skewed
//                            graphs): the centre row stays in registers over a run of equal
//                            centres while the context rows (all distinct within a centre) are
//                            gathered NT at a time with 128-bit loads, scored with the
//                            warp-shaped dot of the SGD kernels and updated with 128-bit
//                            atomics.  HBM-bound: 2 * 4D bytes per triple.
//      glove_train_kernel    the single-warp launch (cfg.deterministic): reproduces
//                            oracle/glove.c bit for bit (explicit round-to-nearest intrinsics,
//                            log / exp from IEEE single operations only).
#include <cub/cub.cuh>

#include <algorithm>

#include "host.cuh"
#include "sgns_device.cuh"

namespace b2e {

constexpr unsigned long long COOC_INVALID = ~0ull;

// ln(x), x > 0 normal: the operation sequence of oracle/glove.c:orc_log_det
__device__ __forceinline__ float log_det(float x) {
    uint32_t u = __float_as_uint(x);
    int e = (int)(u >> 23) - 127;
    float m = __uint_as_float((u & 0x007FFFFFu) | 0x3F800000u);
    if (m > 1.41421356237f) { m = __fmul_rn(m, 0.5f); e += 1; }
    const float s = __fdiv_rn(__fsub_rn(m, 1.0f), __fadd_rn(m, 1.0f));
    const float s2 = __fmul_rn(s, s);
    float p = 1.0f / 9.0f;
    p = __fmaf_rn(p, s2, 1.0f / 7.0f);
    p = __fmaf_rn(p, s2, 1.0f / 5.0f);
    p = __fmaf_rn(p, s2, 1.0f / 3.0f);
    p = __fmaf_rn(p, s2, 1.0f);
    const float lnm = __fmul_rn(__fmul_rn(2.0f, s), p);
    return __fmaf_rn((float)e, 0.693147180559945f, lnm);
}

// slot = (walk, position i, offset d in 1..W): keys of the ordered pairs (i, i+d) and (i+d, i)
__global__ void __launch_bounds__(256) cooc_keys_kernel(const uint32_t *__restrict__ walks, uint64_t n_walks,
                                                        uint32_t L, uint32_t W,
                                                        unsigned long long *__restrict__ keys) {
    const uint64_t total = n_walks * L * W;
    for (uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t d = (uint32_t)(idx % W) + 1u;
        const uint64_t rest = idx / W;
        const uint32_t i = (uint32_t)(rest % L);
        const uint64_t w = rest / L;
        unsigned long long k0 = COOC_INVALID, k1 = COOC_INVALID;
        if (i + d < L) {
            const uint32_t a = __ldg(walks + w * L + i), b = __ldg(walks + w * L + i + d);
            if (a != PAD && b != PAD && a != b) {
                k0 = ((unsigned long long)a << 32) | b;
                k1 = ((unsigned long long)b << 32) | a;
            }
        }
        keys[2 * idx] = k0;
        keys[2 * idx + 1] = k1;
    }
}

__global__ void __launch_bounds__(256) cooc_rowptr_kernel(const unsigned long long *__restrict__ keys,
                                                          uint64_t n_triples, uint64_t n,
                                                          uint64_t *__restrict__ rowptr) {
    const uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v > n) return;
    const unsigned long long target = (unsigned long long)v << 32;
    uint64_t lo = 0, hi = n_triples;
    while (lo < hi) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(keys + mid) < target) lo = mid + 1; else hi = mid;
    }
    rowptr[v] = lo;
}

struct GloveParams {
    const unsigned long long *keys;
    const uint32_t *counts;
    const uint64_t *rowptr;
    uint64_t n;
    uint32_t row_stride, chunks;
    float alpha, clip, lr, max_count;
    float *t0, *t1;
    DeviceCounters *counters;
};

// weight = (x / x_max)^alpha and ln x depend on the count alone: lane s computes them for triple
// base + s of the batch (once, instead of 32 times) and the warp reads them back by shuffle
__device__ __forceinline__ void count_terms(const GloveParams &p, uint64_t base, uint64_t end, uint32_t lane,
                                            float &weight, float &log_count) {
    const float x = base + lane < end ? (float)__ldg(p.counts + base + lane) : 1.0f;
    weight = exp_det(__fmul_rn(p.alpha, log_det(__fdiv_rn(x, p.max_count))));
    log_count = log_det(x);
}

// Single-warp launch (cfg.deterministic): centres in ascending order, the operation sequence of
// oracle/glove.c.  The production launch is glove_tile_kernel below.
template <int CH, int NT>
__global__ void __launch_bounds__(32) glove_train_kernel(const GloveParams p) {
    const uint32_t lane = threadIdx.x & 31u;
    float loss_acc = 0.0f;
    unsigned long long trained = 0;
    for (;;) {
        unsigned long long v = 0;
        if (lane == 0) v = atomicAdd(&p.counters->work_counter, 1ull);
        v = __shfl_sync(FULL, v, 0);
        if (v >= p.n) break;
        const uint64_t begin = __ldg(p.rowptr + v), end = __ldg(p.rowptr + v + 1);
        if (begin == end) continue;
        float *crow = p.t0 + v * p.row_stride;
        float4 h[CH];
        load_row<CH>(crow, p.chunks, lane, h);
        for (uint64_t base = begin; base < end; base += NT) {
            float4 rows[NT][CH];
            uint32_t ids[NT];
#pragma unroll
            for (int s = 0; s < NT; ++s) {  // the contexts of a centre are distinct rows
                const bool on = base + s < end;
                ids[s] = on ? (uint32_t)__ldg(p.keys + base + s) : PAD;
                if (on) load_row<CH>(p.t1 + (uint64_t)ids[s] * p.row_stride, p.chunks, lane, rows[s]);
            }
            float my_weight, my_log;  // lane s < NT holds the two count-only terms of triple s
            count_terms(p, base, end, lane, my_weight, my_log);
#pragma unroll
            for (int s = 0; s < NT; ++s) {
                if (ids[s] == PAD) continue;
                const float f = warp_dot<CH>(h, rows[s]);
                if (fabsf(f) > p.clip) continue;
                const float weight = __shfl_sync(FULL, my_weight, s);
                const float diff = __fsub_rn(f, __shfl_sync(FULL, my_log, s));
                const float g = __fmul_rn(__fmul_rn(__fmul_rn(2.0f, weight), diff), p.lr);
                if (lane == 0) loss_acc += weight * diff * diff;
                ++trained;
                float *target = p.t1 + (uint64_t)ids[s] * p.row_stride;
#pragma unroll
                for (int ch = 0; ch < CH; ++ch) {
                    const float4 old = rows[s][ch];
                    rows[s][ch].x = __fmaf_rn(-g, h[ch].x, old.x);
                    rows[s][ch].y = __fmaf_rn(-g, h[ch].y, old.y);
                    rows[s][ch].z = __fmaf_rn(-g, h[ch].z, old.z);
                    rows[s][ch].w = __fmaf_rn(-g, h[ch].w, old.w);
                    h[ch].x = __fmaf_rn(-g, old.x, h[ch].x);
                    h[ch].y = __fmaf_rn(-g, old.y, h[ch].y);
                    h[ch].z = __fmaf_rn(-g, old.z, h[ch].z);
                    h[ch].w = __fmaf_rn(-g, old.w, h[ch].w);
                }
                store_row<CH>(target, p.chunks, lane, rows[s]);
            }
        }
        store_row<CH>(crow, p.chunks, lane, h);
    }
    if (lane == 0) {
        atomicAdd(&p.counters->pairs, trained);
        atomicAdd(&p.counters->targets, trained);
        atomicAdd(&p.counters->loss_sum, (double)loss_acc);
    }
}

// Production launch.  A hub centre owns a large share of the triples of a skewed graph (R-MAT
// 1 M / 16 M: the pass took as long as the hub's row walked by one warp), so the work unit is a
// TILE of `GLOVE_TILE` consecutive triples of the flat sorted array instead of a centre: every
// warp does the same amount of work whatever the degree distribution.  Inside a tile the warp
// follows the runs of equal centre: at a run boundary it adds `h - h0` (what this run changed)
// to the centre row with one 128-bit atomic per lane -- rows split over several tiles receive
// the sum of their tiles' changes -- and loads the next centre.  Context rows are updated
// with 128-bit atomics too: a context row is shared by many centres trained concurrently and a
// plain read-modify-write would lose all but one of their updates.
constexpr uint32_t GLOVE_TILE = 512;

template <int CH>
__device__ __forceinline__ void flush_centre(float *crow, uint32_t chunks, uint32_t lane, const float4 (&h)[CH],
                                             const float4 (&h0)[CH]) {
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
        const uint32_t c = lane + 32u * ch;
        if (c < chunks)
            atomicAdd(reinterpret_cast<float4 *>(crow + 4u * c),
                      make_float4(h[ch].x - h0[ch].x, h[ch].y - h0[ch].y, h[ch].z - h0[ch].z, h[ch].w - h0[ch].w));
    }
}

template <int CH, int NT>
__global__ void __launch_bounds__(256) glove_tile_kernel(const GloveParams p, uint64_t n_triples) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t n_tiles = (n_triples + GLOVE_TILE - 1) / GLOVE_TILE;
    float loss_acc = 0.0f;
    unsigned long long trained = 0;
    for (;;) {
        unsigned long long tile = 0;
        if (lane == 0) tile = atomicAdd(&p.counters->work_counter, 1ull);
        tile = __shfl_sync(FULL, tile, 0);
        if (tile >= n_tiles) break;
        const uint64_t begin = tile * GLOVE_TILE, end = min(begin + GLOVE_TILE, n_triples);
        uint32_t centre = PAD;
        float4 h[CH], h0[CH];
        for (uint64_t base = begin; base < end; base += NT) {
            float4 rows[NT][CH];
            uint32_t ids[NT], cen[NT];
#pragma unroll
            for (int s = 0; s < NT; ++s) {
                const bool on = base + s < end;
                const unsigned long long key = on ? __ldg(p.keys + base + s) : ~0ull;
                ids[s] = on ? (uint32_t)key : PAD;
                cen[s] = (uint32_t)(key >> 32);
                if (on) load_row<CH>(p.t1 + (uint64_t)ids[s] * p.row_stride, p.chunks, lane, rows[s]);
            }
            float my_weight, my_log;
            count_terms(p, base, end, lane, my_weight, my_log);
#pragma unroll
            for (int s = 0; s < NT; ++s) {
                if (ids[s] == PAD) continue;
                if (cen[s] != centre) {  // run boundary (warp-uniform)
                    if (centre != PAD) flush_centre<CH>(p.t0 + (uint64_t)centre * p.row_stride, p.chunks, lane, h, h0);
                    centre = cen[s];
                    load_row<CH>(p.t0 + (uint64_t)centre * p.row_stride, p.chunks, lane, h);
#pragma unroll
                    for (int ch = 0; ch < CH; ++ch) h0[ch] = h[ch];
                }
                const float f = warp_dot<CH>(h, rows[s]);
                if (fabsf(f) > p.clip) continue;
                const float weight = __shfl_sync(FULL, my_weight, s);
                const float diff = __fsub_rn(f, __shfl_sync(FULL, my_log, s));
                const float g = __fmul_rn(__fmul_rn(__fmul_rn(2.0f, weight), diff), p.lr);
                if (lane == 0) loss_acc += weight * diff * diff;
                ++trained;
                float *target = p.t1 + (uint64_t)ids[s] * p.row_stride;
#pragma unroll
                for (int ch = 0; ch < CH; ++ch) {
                    const float4 old = rows[s][ch];
                    const uint32_t c = lane + 32u * ch;
                    if (c < p.chunks)
                        atomicAdd(reinterpret_cast<float4 *>(target + 4u * c),
                                  make_float4(-g * h[ch].x, -g * h[ch].y, -g * h[ch].z, -g * h[ch].w));
                    h[ch].x = __fmaf_rn(-g, old.x, h[ch].x);
                    h[ch].y = __fmaf_rn(-g, old.y, h[ch].y);
                    h[ch].z = __fmaf_rn(-g, old.z, h[ch].z);
                    h[ch].w = __fmaf_rn(-g, old.w, h[ch].w);
                }
            }
        }
        if (centre != PAD) flush_centre<CH>(p.t0 + (uint64_t)centre * p.row_stride, p.chunks, lane, h, h0);
    }
    if (lane == 0) {
        atomicAdd(&p.counters->pairs, trained);
        atomicAdd(&p.counters->targets, trained);
        atomicAdd(&p.counters->loss_sum, (double)loss_acc);
    }
}

template <int CH, int NT>
static cudaError_t launch_glove_one(const GloveParams &p, uint64_t n_triples, bool deterministic, int sm_count,
                                    uint64_t max_warps, cudaStream_t stream) {
    cudaError_t err = cudaMemsetAsync(&p.counters->work_counter, 0, sizeof(unsigned long long), stream);
    if (err != cudaSuccess) return err;
    if (deterministic) {
        glove_train_kernel<CH, NT><<<1, 32, 0, stream>>>(p);
        return cudaGetLastError();
    }
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, glove_tile_kernel<CH, NT>, 256, 0);
    if (err != cudaSuccess) return err;
    uint64_t grid = (uint64_t)sm_count * std::max(per_sm, 1);  // persistent, tiles fetched dynamically
    const uint64_t n_tiles = (n_triples + GLOVE_TILE - 1) / GLOVE_TILE;
    grid = std::max<uint64_t>(1, std::min<uint64_t>(grid, (std::min<uint64_t>(n_tiles, max_warps) + 7) / 8));
    glove_tile_kernel<CH, NT><<<(unsigned)grid, 256, 0, stream>>>(p, n_triples);
    return cudaGetLastError();
}

// walks per co-occurrence chunk: at most 2^27 key slots (1 GiB of keys, sorted out of place)
uint64_t glove_chunk_walks(uint32_t walk_length, uint32_t window) {
    const uint64_t slots_per_walk = 2ull * walk_length * window;
    return std::max<uint64_t>(1, (1ull << 27) / slots_per_walk);
}

// Adds the co-occurrences of `n_walks` device-resident walks to the state (merged by key).
cudaError_t glove_accumulate(GloveState &g, const uint32_t *d_walks, uint64_t n_walks, uint32_t L,
                             uint32_t W, cudaStream_t stream, std::string &error) {
    typedef unsigned long long u64;
    const uint64_t slots = 2ull * n_walks * L * W;
    if (slots == 0) return cudaSuccess;
    CUDA_CHECK(g.d_scratch_keys.reserve(2 * slots * sizeof(u64)));
    u64 *raw = g.d_scratch_keys.get(), *sorted = g.d_scratch_keys.get() + slots;
    const uint64_t grid = std::min<uint64_t>((slots / 2 + 255) / 256, 148ull * 32);
    cooc_keys_kernel<<<(unsigned)grid, 256, 0, stream>>>(d_walks, n_walks, L, W, raw);
    CUDA_CHECK(cudaGetLastError());

    size_t need = 0, bytes = 0;
    CUDA_CHECK(cub::DeviceRadixSort::SortKeys(nullptr, bytes, raw, sorted, slots, 0, 64, stream));
    need = bytes;
    // run-length encode into the tail of the merge buffers (sized below)
    const uint64_t merged_cap = g.n_triples + slots;
    CUDA_CHECK(g.d_merge_keys.reserve(2 * merged_cap * sizeof(u64)));
    CUDA_CHECK(g.d_merge_counts.reserve(2 * merged_cap * sizeof(uint32_t)));
    CUDA_CHECK(g.d_scalar.reserve(16));
    u64 *cat_keys = g.d_merge_keys.get(), *out_keys = g.d_merge_keys.get() + merged_cap;
    uint32_t *cat_counts = g.d_merge_counts.get(), *out_counts = g.d_merge_counts.get() + merged_cap;
    uint64_t *d_runs = reinterpret_cast<uint64_t *>(g.d_scalar.get());
    CUDA_CHECK(cub::DeviceRunLengthEncode::Encode(nullptr, bytes, sorted, cat_keys + g.n_triples,
                                                 cat_counts + g.n_triples, d_runs, slots, stream));
    need = std::max(need, bytes);
    // merging two sorted lists is one linear pass (sorting the concatenation would be eight)
    CUDA_CHECK(cub::DeviceMerge::MergePairs(nullptr, bytes, g.d_keys.get(), g.d_counts.get(), (int64_t)g.n_triples,
                                           cat_keys + g.n_triples, cat_counts + g.n_triples, (int64_t)slots,
                                           out_keys, out_counts, ::cuda::std::less<>{}, stream));
    need = std::max(need, bytes);
    CUDA_CHECK(cub::DeviceReduce::ReduceByKey(nullptr, bytes, out_keys, cat_keys, out_counts, cat_counts, d_runs,
                                             cub::Sum(), merged_cap, stream));
    need = std::max(need, bytes);
    CUDA_CHECK(g.d_temp.reserve(need));

    bytes = g.d_temp.bytes();
    CUDA_CHECK(cub::DeviceRadixSort::SortKeys(g.d_temp.get(), bytes, raw, sorted, slots, 0, 64, stream));
    // the chunk's (key, count) list goes behind the room of the triples gathered so far
    bytes = g.d_temp.bytes();
    CUDA_CHECK(cub::DeviceRunLengthEncode::Encode(g.d_temp.get(), bytes, sorted, cat_keys + g.n_triples,
                                                 cat_counts + g.n_triples, d_runs, slots, stream));
    uint64_t runs = 0;
    CUDA_CHECK(cudaMemcpyAsync(&runs, d_runs, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    if (runs) {  // the all-ones key, if present, is the last run
        u64 last = 0;
        CUDA_CHECK(cudaMemcpyAsync(&last, cat_keys + g.n_triples + runs - 1, sizeof(u64), cudaMemcpyDeviceToHost, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
        if (last == COOC_INVALID) --runs;
    }
    if (runs == 0) return cudaSuccess;  // nothing new: the resident triples stand
    uint64_t total = runs;
    const u64 *result_keys = cat_keys;  // g.n_triples == 0: the chunk's list is the result
    const uint32_t *result_counts = cat_counts;
    if (g.n_triples) {  // both lists are sorted: merge, then add the counts of equal keys
        total = g.n_triples + runs;
        bytes = g.d_temp.bytes();
        CUDA_CHECK(cub::DeviceMerge::MergePairs(g.d_temp.get(), bytes, g.d_keys.get(), g.d_counts.get(), (int64_t)g.n_triples,
                                               cat_keys + g.n_triples, cat_counts + g.n_triples, (int64_t)runs,
                                               out_keys, out_counts, ::cuda::std::less<>{}, stream));
        bytes = g.d_temp.bytes();
        CUDA_CHECK(cub::DeviceReduce::ReduceByKey(g.d_temp.get(), bytes, out_keys, cat_keys, out_counts, cat_counts,
                                                 d_runs, cub::Sum(), total, stream));
        CUDA_CHECK(cudaMemcpyAsync(&total, d_runs, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
    }
    CUDA_CHECK(g.d_keys.reserve(total * sizeof(u64)));
    CUDA_CHECK(g.d_counts.reserve(total * sizeof(uint32_t)));
    CUDA_CHECK(cudaMemcpyAsync(g.d_keys.get(), result_keys, total * sizeof(u64), cudaMemcpyDeviceToDevice, stream));
    CUDA_CHECK(cudaMemcpyAsync(g.d_counts.get(), result_counts, total * sizeof(uint32_t), cudaMemcpyDeviceToDevice, stream));
    g.n_triples = total;
    g.finalised = false;
    return cudaSuccess;
}

// row offsets by centre and the largest count: needed before training
cudaError_t glove_finalise(GloveState &g, uint64_t n, cudaStream_t stream, std::string &error) {
    CUDA_CHECK(g.d_rowptr.reserve((n + 1) * sizeof(uint64_t)));
    cooc_rowptr_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, stream>>>(g.d_keys.get(), g.n_triples, n, g.d_rowptr.get());
    CUDA_CHECK(cudaGetLastError());
    g.max_count = 1;
    if (g.n_triples) {
        CUDA_CHECK(g.d_scalar.reserve(16));
        uint32_t *d_max = reinterpret_cast<uint32_t *>(g.d_scalar.get());
        size_t bytes = 0;
        CUDA_CHECK(cub::DeviceReduce::Max(nullptr, bytes, g.d_counts.get(), d_max, g.n_triples, stream));
        CUDA_CHECK(g.d_temp.reserve(bytes));
        bytes = g.d_temp.bytes();
        CUDA_CHECK(cub::DeviceReduce::Max(g.d_temp.get(), bytes, g.d_counts.get(), d_max, g.n_triples, stream));
        CUDA_CHECK(cudaMemcpyAsync(&g.max_count, d_max, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    }
    CUDA_CHECK(cudaStreamSynchronize(stream));
    g.finalised = true;
    return cudaSuccess;
}

cudaError_t glove_train(const GloveState &g, uint64_t n, uint32_t row_stride, uint32_t embedding_size,
                        float alpha, float clip, float lr, float *t0, float *t1, DeviceCounters *counters,
                        bool deterministic, int sm_count, uint64_t max_warps, cudaStream_t stream) {
    if (g.n_triples == 0) return cudaSuccess;
    GloveParams p;
    p.keys = g.d_keys.get();
    p.counts = g.d_counts.get();
    p.rowptr = g.d_rowptr.get();
    p.n = n;
    p.row_stride = row_stride;
    p.chunks = (embedding_size + 3u) / 4u;
    p.alpha = alpha;
    p.clip = clip;
    p.lr = lr;
    p.max_count = (float)g.max_count;
    p.t0 = t0;
    p.t1 = t1;
    p.counters = counters;
    // 4 rows per batch: 64 registers, 4 CTAs per SM -- 6.0 G triples/s against 3.8 G with 8 rows
    // (95 registers, 2 CTAs per SM) on R-MAT 1 M / 16 M
    if (p.chunks <= 32) return launch_glove_one<1, 4>(p, g.n_triples, deterministic, sm_count, max_warps, stream);
    if (p.chunks <= 64) return launch_glove_one<2, 4>(p, g.n_triples, deterministic, sm_count, max_warps, stream);
    if (p.chunks <= 128) return launch_glove_one<4, 2>(p, g.n_triples, deterministic, sm_count, max_warps, stream);
    return cudaErrorInvalidValue;
}

// ---- co-occurrence by centre range: the way past 2^31 key slots per epoch ----
//
// The reference's GloVe defaults (walk_length = 512, window_size = 5, node2vec_glove.py:8-30) emit
// 5 120 key slots per start node and epoch: beyond ~0.4 M nodes an epoch's co-occurrence no
// longer fits one sort.  Every key (centre, context) belongs to exactly one centre, so the
// epoch is cut into ranges of centre ids: the occurrences of the epoch's walks are bucketed by
// range once (one counting pass, one scatter pass), and each range is then counted (emit ->
// sort -> run-length encode) and trained on its own, in ascending order of centre -- the exact
// counts and the exact order of the one-piece path, for any number of ranges.

// tokens per node over the walks of an epoch
__global__ void __launch_bounds__(256) token_histogram_kernel(const uint32_t *__restrict__ walks, uint64_t tokens,
                                                              uint32_t *__restrict__ histogram) {
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < tokens;
         p += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t v = __ldg(walks + p);
        if (v != PAD) atomicAdd(histogram + v, 1u);
    }
}

// position p of a walk token goes to the range that holds its node: bounds[r] <= node < bounds[r + 1];
// tokens of nodes outside [bounds[0], bounds[ranges]) (centres another rank owns) are skipped
__global__ void __launch_bounds__(256) bucket_positions_kernel(const uint32_t *__restrict__ walks, uint64_t tokens,
                                                               const uint32_t *__restrict__ bounds, uint32_t ranges,
                                                               unsigned long long *__restrict__ cursor,
                                                               unsigned long long *__restrict__ positions) {
    const uint32_t first = __ldg(bounds), last = __ldg(bounds + ranges);
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < tokens;
         p += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t v = __ldg(walks + p);
        if (v == PAD || v < first || v >= last) continue;
        uint32_t lo = 0, hi = ranges;  // last r with bounds[r] <= v
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (__ldg(bounds + mid) <= v) lo = mid; else hi = mid;
        }
        positions[atomicAdd(cursor + lo, 1ull)] = p;
    }
}

// occurrence (position p) x window offset: the key (centre, context) or the all-ones key
__global__ void __launch_bounds__(256) range_keys_kernel(const uint32_t *__restrict__ walks, uint32_t L, uint32_t W,
                                                         const unsigned long long *__restrict__ positions,
                                                         uint64_t count, unsigned long long *__restrict__ keys) {
    const uint64_t total = count * 2ull * W;
    for (uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t occurrence = idx / (2u * W);
        const uint32_t slot = (uint32_t)(idx - occurrence * 2u * W);
        const uint32_t d = (slot >> 1) + 1u;
        const unsigned long long p = __ldg(positions + occurrence);
        const uint32_t i = (uint32_t)(p % L);
        const long long j = (slot & 1u) ? (long long)i - d : (long long)i + d;
        unsigned long long key = COOC_INVALID;
        if (j >= 0 && j < (long long)L) {
            const uint32_t a = __ldg(walks + p), b = __ldg(walks + (p - i) + (uint64_t)j);
            if (b != PAD && a != b) key = ((unsigned long long)a << 32) | b;
        }
        keys[idx] = key;
    }
}

cudaError_t glove_token_histogram(const uint32_t *d_walks, uint64_t tokens, uint32_t *d_histogram, uint64_t n,
                                  cudaStream_t stream) {
    const cudaError_t e = cudaMemsetAsync(d_histogram, 0, n * sizeof(uint32_t), stream);
    if (e != cudaSuccess || tokens == 0) return e;
    token_histogram_kernel<<<148 * 16, 256, 0, stream>>>(d_walks, tokens, d_histogram);
    return cudaGetLastError();
}

cudaError_t glove_bucket_positions(const uint32_t *d_walks, uint64_t tokens, const uint32_t *d_bounds, uint32_t ranges,
                                   unsigned long long *d_cursor, unsigned long long *d_positions,
                                   cudaStream_t stream) {
    if (tokens == 0) return cudaSuccess;
    bucket_positions_kernel<<<148 * 16, 256, 0, stream>>>(d_walks, tokens, d_bounds, ranges, d_cursor, d_positions);
    return cudaGetLastError();
}

// The co-occurrence triples of one centre range replace the resident ones (g.n_triples, sorted
// by (centre, context)); `count` occurrences, 2 W key slots each.
cudaError_t glove_range_triples(GloveState &g, const uint32_t *d_walks, uint32_t L, uint32_t W,
                                const unsigned long long *d_positions, uint64_t count, cudaStream_t stream,
                                std::string &error) {
    typedef unsigned long long u64;
    g.n_triples = 0;
    g.finalised = false;
    const uint64_t slots = count * 2ull * W;
    if (slots == 0) return cudaSuccess;
    CUDA_CHECK(g.d_scratch_keys.reserve(2 * slots * sizeof(u64)));
    u64 *raw = g.d_scratch_keys.get(), *sorted = g.d_scratch_keys.get() + slots;
    const uint64_t grid = std::min<uint64_t>((slots + 255) / 256, 148ull * 32);
    range_keys_kernel<<<(unsigned)grid, 256, 0, stream>>>(d_walks, L, W, d_positions, count, raw);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(g.d_keys.reserve(slots * sizeof(u64)));
    CUDA_CHECK(g.d_counts.reserve(slots * sizeof(uint32_t)));
    CUDA_CHECK(g.d_scalar.reserve(16));
    uint64_t *d_runs = reinterpret_cast<uint64_t *>(g.d_scalar.get());
    size_t bytes = 0, need = 0;
    CUDA_CHECK(cub::DeviceRadixSort::SortKeys(nullptr, bytes, raw, sorted, slots, 0, 64, stream));
    need = bytes;
    CUDA_CHECK(cub::DeviceRunLengthEncode::Encode(nullptr, bytes, sorted, g.d_keys.get(), g.d_counts.get(), d_runs, slots, stream));
    need = std::max(need, bytes);
    CUDA_CHECK(g.d_temp.reserve(need));
    bytes = g.d_temp.bytes();
    CUDA_CHECK(cub::DeviceRadixSort::SortKeys(g.d_temp.get(), bytes, raw, sorted, slots, 0, 64, stream));
    bytes = g.d_temp.bytes();
    CUDA_CHECK(cub::DeviceRunLengthEncode::Encode(g.d_temp.get(), bytes, sorted, g.d_keys.get(), g.d_counts.get(), d_runs, slots, stream));
    uint64_t runs = 0;
    CUDA_CHECK(cudaMemcpyAsync(&runs, d_runs, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    if (runs) {  // the all-ones key, if present, is the last run
        u64 last = 0;
        CUDA_CHECK(cudaMemcpyAsync(&last, g.d_keys.get() + runs - 1, sizeof(u64), cudaMemcpyDeviceToHost, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
        if (last == COOC_INVALID) --runs;
    }
    g.n_triples = runs;
    return cudaSuccess;
}

// largest count of the resident triples (0 when there are none)
cudaError_t glove_max_count(GloveState &g, uint32_t *max_count, cudaStream_t stream, std::string &error) {
    *max_count = 0;
    if (g.n_triples == 0) return cudaSuccess;
    CUDA_CHECK(g.d_scalar.reserve(16));
    uint32_t *d_max = reinterpret_cast<uint32_t *>(g.d_scalar.get());
    size_t bytes = 0;
    CUDA_CHECK(cub::DeviceReduce::Max(nullptr, bytes, g.d_counts.get(), d_max, g.n_triples, stream));
    CUDA_CHECK(g.d_temp.reserve(bytes));
    bytes = g.d_temp.bytes();
    CUDA_CHECK(cub::DeviceReduce::Max(g.d_temp.get(), bytes, g.d_counts.get(), d_max, g.n_triples, stream));
    CUDA_CHECK(cudaMemcpyAsync(max_count, d_max, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    return cudaSuccess;
}

}  // namespace b2e
