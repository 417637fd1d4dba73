// Shared device helpers and the handle layout of the B200 engine (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/b2e.h"

namespace b2e {

// Philox stream tags (top byte of counter word 3); the normative layout is in DESIGN.md.
constexpr uint32_t TAG_WALK1 = 1u;  // first-order steps, 4 per block
constexpr uint32_t TAG_WALK2 = 2u;  // second-order trials, 2 per block
constexpr uint32_t TAG_NEG = 3u;    // negative draws
constexpr uint32_t TAG_INIT0 = 4u;  // table 0 initialisation
constexpr uint32_t TAG_INIT1 = 5u;  // table 1 initialisation
constexpr uint32_t TAG_WALK3 = 7u;  // general walks (normalize_by_degree, typed): 1 trial per block
constexpr uint32_t TAG_SKIP = 6u;   // stochastic_downsample_by_degree, one draw per centre
constexpr uint32_t TAG_FOLD = 12u;  // second-order trials with the return edge folded: 1 trial per block
constexpr uint32_t MAX_TRIALS = 1u << 20;
constexpr uint32_t PAD = B2E_PAD_TOKEN;

__device__ __forceinline__ uint4 philox4x32_10(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1,
                                               uint32_t c2, uint32_t c3) {
#pragma unroll
    for (int round = 0; round < 10; ++round) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

struct DeviceCounters {
    unsigned long long walk_steps;
    unsigned long long walk_trials;
    unsigned long long walk_searches;
    unsigned long long walk_probes;         // gathers spent on adjacency checks (filter words, row bounds, bisection)
    unsigned long long walk_filter_rejects; // adjacency checks answered "not a neighbour" by the row filter alone
    unsigned long long pairs;
    unsigned long long targets;
    double loss_sum;
    unsigned long long work_counter;  // dynamic walk fetch of the SGD kernels
};

struct WalkParams {
    const int64_t *indptr;
    const uint32_t *indices;
    const uint2 *edge_alias;  // per-row alias tables of a weighted graph ({thr, alias} per edge), or nullptr
    const uint32_t *node_types, *edge_types;  // [n] / [nnz] type ids of typed walks, or nullptr
    unsigned long long q_node[2], q_edge[2];  // accept thresholds [same type, changed type]
    const uint32_t *sources;
    uint64_t n_src;
    uint32_t seed_lo, seed_hi;
    uint64_t first_walk, n_walks, walk_id_stride;
    uint32_t walk_length;
    unsigned long long thr_return, thr_common, thr_explore;
    uint32_t *out;
    DeviceCounters *counters;
    uint32_t undirected;     // every edge has its mirror (verified at load): allows the short-row check
    const unsigned long long *filter;  // per-row blocked Bloom filters over the neighbour lists, or nullptr
    unsigned long long fold_excess;    // E > 0: the return edge is folded out of the envelope (TAG_FOLD)
    int sm_count;
};

struct TrainParams {
    const uint32_t *walks;
    uint64_t first_walk, n_walks, walk_id_stride;
    uint32_t seed_lo, seed_hi;
    uint32_t n;
    uint32_t walk_length, window, negatives;
    uint32_t row_stride;  // floats between rows in HBM: rows start on 128 B lines
    uint32_t chunks;      // float4 chunks of a row that hold data: ceil(embedding_size / 4)
    float clip, lr, inv_scale;
    uint32_t use_alias, normalize_lr, scale_dot;
    uint32_t downsample;  // stochastic_downsample_by_degree: max degree + 1, 0 = off
    uint32_t shared_negatives;  // SkipGram: one set of negatives per centre (skipgram_shared_kernel)
    const uint2 *alias;  // {threshold, alias} per node
    const int64_t *indptr;
    float *t0, *t1;
    DeviceCounters *counters;
};

cudaError_t launch_walks(const WalkParams &p, bool second_order, cudaStream_t stream);
cudaError_t launch_walklet_split(const uint32_t *raw, uint64_t n_walks, uint32_t walk_length, uint32_t scale,
                                 uint32_t *out, cudaStream_t stream);
cudaError_t launch_symmetry_check(const int64_t *indptr, const uint32_t *indices, uint64_t n,
                                  uint64_t nnz, int *d_flag, cudaStream_t stream);
// *d_flags |= 1: a destination id >= n; |= 2: a row that is not strictly ascending
cudaError_t launch_csr_check(const int64_t *indptr, const uint32_t *indices, uint64_t n, int *d_flags,
                             int sm_count, cudaStream_t stream);
// alias_build.cu: offsets check (*d_flags |= 4), start nodes + maximum degree + alias table on the device
cudaError_t check_indptr_device(const int64_t *d_indptr, uint64_t n, uint64_t nnz, int *d_flags, cudaStream_t stream);
cudaError_t build_node_tables(const int64_t *d_indptr, const int64_t *host_indptr, uint64_t n, double alpha,
                              uint32_t *d_sources, uint64_t *n_src_out, uint64_t *max_degree_out, uint2 *d_table,
                              cudaStream_t stream, std::string &error);
// alias_build.cu: the per-row alias tables of a weighted graph, {thr, alias index inside the row} per
// edge, bit-identical to oracle/walks.c (orc_edge_alias); *longest_row: the largest degree
cudaError_t build_edge_alias(const int64_t *d_indptr, const float *d_weights, uint64_t n, uint64_t nnz,
                             uint2 *d_table, uint64_t *longest_row, cudaStream_t stream, std::string &error);
// normalize_by_degree: out[e] = (weights ? weights[e] : 1) / max(deg(indices[e]), 1), in float32
cudaError_t launch_degree_normalise(const int64_t *d_indptr, const uint32_t *d_indices, const float *d_weights,
                                    uint64_t nnz, float *d_out, cudaStream_t stream);
uint64_t row_filter_words(uint64_t nnz);
cudaError_t launch_row_filter_build(const int64_t *indptr, const uint32_t *indices, uint64_t n,
                                    unsigned long long *filter, int sm_count, cudaStream_t stream);
cudaError_t launch_exchange_average(float *const t0[], float *const t1[], uint32_t world, uint32_t rank,
                                    uint64_t n, uint32_t row_stride, uint32_t chunks, int sm_count,
                                    cudaStream_t stream);
// GloVe's merge of a sharded epoch: every replica takes row v of T0 from the replica of its owner
// and T1 = snapshot + sum over the ranks of (T1_g - snapshot); this rank reduces the rows
// [n rank / world, n (rank + 1) / world)
cudaError_t launch_glove_merge(float *const t0[], float *const t1[], const float *snapshot,
                               const uint32_t *owner_bounds, uint32_t world, uint32_t rank, uint64_t n,
                               uint32_t row_stride, uint32_t chunks, int sm_count, cudaStream_t stream);
cudaError_t launch_pack_rows(const float *table, uint64_t rows, uint32_t row_stride, uint32_t dim, float *dense,
                             int sm_count, cudaStream_t stream);
cudaError_t launch_tables_digest(const float *t0, const float *t1, uint64_t n, uint32_t row_stride,
                                 uint32_t dim, void *d_out, int sm_count, cudaStream_t stream);
cudaError_t launch_init_tables(float *t0, float *t1, uint64_t n, uint32_t embedding_size,
                               uint32_t row_stride, uint64_t seed, cudaStream_t stream);
// max_warps caps how many walks are trained concurrently (Hogwild staleness on small graphs)
cudaError_t launch_train(const TrainParams &p, uint32_t model, bool deterministic, int sm_count,
                         uint64_t max_warps, cudaStream_t stream);
bool pipe_supported(const TrainParams &p, uint32_t model);
bool shared_negatives_supported(const TrainParams &p);
cudaError_t launch_train_pipe(const TrainParams &p, uint32_t model, bool deterministic, int sm_count,
                              uint64_t max_warps, cudaStream_t stream);

}  // namespace b2e
