// The step after the embedding path (SURVEY.md 8(f) row 4) for sm_100a: edge embeddings and a
// perceptron edge scorer computed from node features that stay resident in HBM.
//
// Replaces, for this step,
//   * `EdgeTransformer.transform` -- the twelve numpy methods of
//     /root/reference/embiggen/embedding_transformers/edge_transformer.py:12-361;
//   * `models.EdgePredictionPerceptron` behind `PerceptronEdgePrediction`
//     (/root/reference/embiggen/edge_prediction/edge_prediction_ensmallen/perceptron.py:15-300):
//     fit (Adam, scale-free negative sampling) and predict_proba.
// Normative recipe and parity status: oracle/edge_prediction.py.
//
// All three kernels are row gathers (HBM / L2 bound, like the SGD kernels): one warp per edge,
// lane l reads elements l, l + 32, ... of the two node rows (coalesced 128 B requests).  The
// training step never materialises the edge embedding: features are recomputed from the two
// rows in registers for the forward dot and again for the gradient, the gradient is reduced
// per CTA in shared memory and flushed with one atomicAdd per feature, and a second tiny kernel
// applies Adam.  Elementwise methods are single IEEE operations (bit-exact against numpy); the
// two scalar methods reduce over the warp (last-ulp differences from numpy's pairwise sums).
#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "host.cuh"

namespace b2e {

constexpr uint32_t TAG_EDGE_SAMPLE = 8u;
constexpr uint32_t TAG_PERCEPTRON_INIT = 9u;
constexpr int MAX_METHODS = 12;

constexpr int MAX_METRICS = 5;

struct MethodList {
    uint32_t n;
    uint32_t id[MAX_METHODS];
    uint32_t offset[MAX_METHODS];  // first feature of the method in the concatenation
    uint32_t n_metrics;            // topological edge features, after the edge embeddings
    uint32_t metric_id[MAX_METRICS];
    uint32_t metric_offset[MAX_METRICS];
    uint32_t size;                 // total number of features
};

// what the topological edge features read: the support graph's sorted CSR
struct GraphView {
    const int64_t *indptr;
    const uint32_t *indices;
    float inv_max_degree;
};

__host__ __device__ __forceinline__ uint32_t method_width(uint32_t id, uint32_t dim) {
    return id == B2E_EDGE_CONCATENATE ? 2u * dim
                                      : (id == B2E_EDGE_L2_DISTANCE || id == B2E_EDGE_COSINE_SIMILARITY) ? 1u : dim;
}

__device__ __forceinline__ float elementwise(uint32_t id, float a, float b) {
    switch (id) {
        case B2E_EDGE_HADAMARD: return __fmul_rn(a, b);
        case B2E_EDGE_SUM: return __fadd_rn(a, b);
        case B2E_EDGE_AVERAGE: return __fdiv_rn(__fadd_rn(a, b), 2.0f);
        case B2E_EDGE_L1: return __fsub_rn(a, b);
        case B2E_EDGE_ABSOLUTE_L1: return fabsf(__fsub_rn(a, b));
        case B2E_EDGE_SQUARED_L2: { const float d = __fsub_rn(a, b); return __fmul_rn(d, d); }
        case B2E_EDGE_L2: { const float d = __fsub_rn(a, b); return __fsqrt_rn(__fmul_rn(d, d)); }
        case B2E_EDGE_MIN: return fminf(a, b);
        default: return fmaxf(a, b);  // B2E_EDGE_MAX
    }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// the two scalar methods of an edge: L2 distance and cosine similarity (norm clamped at 1e-6,
// edge_transformer.py:263-272)
__device__ __forceinline__ void scalar_features(const float *__restrict__ a, const float *__restrict__ b,
                                                uint32_t dim, uint32_t lane, float &l2, float &cosine) {
    float dd = 0.f, ab = 0.f, aa = 0.f, bb = 0.f;
    for (uint32_t j = lane; j < dim; j += 32u) {
        const float x = __ldg(a + j), y = __ldg(b + j), d = x - y;
        dd = fmaf(d, d, dd);
        ab = fmaf(x, y, ab);
        aa = fmaf(x, x, aa);
        bb = fmaf(y, y, bb);
    }
    dd = warp_sum(dd); ab = warp_sum(ab); aa = warp_sum(aa); bb = warp_sum(bb);
    l2 = sqrtf(dd);
    float norm = sqrtf(aa) * sqrtf(bb);
    if (norm < 1e-6f) norm = 1e-6f;
    cosine = ab / norm;
}

// ---- topological edge features (perceptron.py:38-46): one pass over the common neighbours ----
// values: [0] deg(u) / max degree, [1] deg(v) / max degree, [2] Adamic-Adar, [3] Jaccard,
// [4] resource allocation index, [5] preferential attachment (normalised by max degree^2).
// Lanes stride over the shorter row and bisect the longer one.
__device__ __forceinline__ void finish_metric_values(const GraphView &g, float du, float dv, float common,
                                                     float adamic_adar, float resource, float (&out)[6]) {
    const float uni = du + dv - common;
    out[0] = du * g.inv_max_degree;
    out[1] = dv * g.inv_max_degree;
    out[2] = adamic_adar;
    out[3] = uni > 0.f ? common / uni : 0.f;
    out[4] = resource;
    out[5] = (du * g.inv_max_degree) * (dv * g.inv_max_degree);
}

__device__ __forceinline__ void edge_metric_values(const GraphView &g, uint32_t u, uint32_t v, uint32_t lane,
                                                   float (&out)[6]) {
    int64_t a_off = __ldg(g.indptr + u), b_off = __ldg(g.indptr + v);
    uint32_t a_len = (uint32_t)(__ldg(g.indptr + u + 1) - a_off), b_len = (uint32_t)(__ldg(g.indptr + v + 1) - b_off);
    const float du = (float)a_len, dv = (float)b_len;
    if (a_len > b_len) {
        const int64_t t = a_off; a_off = b_off; b_off = t;
        const uint32_t l = a_len; a_len = b_len; b_len = l;
    }
    float common = 0.f, adamic_adar = 0.f, resource = 0.f;
    uint32_t from = 0;  // a lane's successive keys ascend: its lower bounds do too
    for (uint32_t i = lane; i < a_len; i += 32u) {
        const uint32_t x = __ldg(g.indices + a_off + i);
        // gallop from the previous lower bound, then bisect the bracket: O(log gap) probes
        // instead of O(log deg), which is what makes hub-hub pairs (the bulk of a scale-free
        // mini-batch) affordable
        uint32_t lo = from, step = 1;
        while (lo + step < b_len && __ldg(g.indices + b_off + lo + step) < x) {
            lo += step;
            step <<= 1;
        }
        uint32_t hi = min(lo + step, b_len);
        while (lo < hi) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            if (__ldg(g.indices + b_off + mid) < x) lo = mid + 1; else hi = mid;
        }
        from = lo;
        if (lo < b_len && __ldg(g.indices + b_off + lo) == x) {
            const float dx = (float)(uint32_t)(__ldg(g.indptr + x + 1) - __ldg(g.indptr + x));
            common += 1.f;
            if (dx > 1.f) adamic_adar += 1.f / logf(dx);
            if (dx > 0.f) resource += 1.f / dx;
        }
    }
    common = warp_sum(common);
    adamic_adar = warp_sum(adamic_adar);
    resource = warp_sum(resource);
    finish_metric_values(g, du, dv, common, adamic_adar, resource, out);
}

// The same pass by a whole CTA for the `count` samples its warps drew (perceptron_step_kernel):
// a scale-free mini-batch is full of hub-hub negatives whose two rows are long, and a step lasts
// as long as its slowest sample, so all 256 threads stride over the shorter row of one sample
// after the other.  sums[s] = {common, Adamic-Adar, resource allocation} of sample s.
__device__ __forceinline__ void cta_common_neighbours(const GraphView &g, const uint32_t *s_u, const uint32_t *s_v,
                                                      const uint32_t *s_valid, uint32_t count, float (*sums)[3]) {
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t s = 0; s < count; ++s) {
        if (!s_valid[s]) continue;  // CTA-uniform
        int64_t a_off = __ldg(g.indptr + s_u[s]), b_off = __ldg(g.indptr + s_v[s]);
        uint32_t a_len = (uint32_t)(__ldg(g.indptr + s_u[s] + 1) - a_off);
        uint32_t b_len = (uint32_t)(__ldg(g.indptr + s_v[s] + 1) - b_off);
        if (a_len > b_len) {
            const int64_t t = a_off; a_off = b_off; b_off = t;
            const uint32_t l = a_len; a_len = b_len; b_len = l;
        }
        float common = 0.f, adamic_adar = 0.f, resource = 0.f;
        uint32_t from = 0;
        for (uint32_t i = threadIdx.x; i < a_len; i += blockDim.x) {
            const uint32_t x = __ldg(g.indices + a_off + i);
            uint32_t lo = from, step = 1;
            while (lo + step < b_len && __ldg(g.indices + b_off + lo + step) < x) {
                lo += step;
                step <<= 1;
            }
            uint32_t hi = min(lo + step, b_len);
            while (lo < hi) {
                const uint32_t mid = lo + ((hi - lo) >> 1);
                if (__ldg(g.indices + b_off + mid) < x) lo = mid + 1; else hi = mid;
            }
            from = lo;
            if (lo < b_len && __ldg(g.indices + b_off + lo) == x) {
                const float dx = (float)(uint32_t)(__ldg(g.indptr + x + 1) - __ldg(g.indptr + x));
                common += 1.f;
                if (dx > 1.f) adamic_adar += 1.f / logf(dx);
                if (dx > 0.f) resource += 1.f / dx;
            }
        }
        if (a_len > (threadIdx.x & ~31u)) {  // warp-uniform: warps past the end of the row have nothing to add
            common = warp_sum(common);
            adamic_adar = warp_sum(adamic_adar);
            resource = warp_sum(resource);
            if (lane == 0 && common > 0.f) {
                atomicAdd(&sums[s][0], common);
                atomicAdd(&sums[s][1], adamic_adar);
                atomicAdd(&sums[s][2], resource);
            }
        }
    }
}

__device__ __forceinline__ uint32_t metric_slot(uint32_t id) {  // first value of the metric in `out`
    return id == B2E_EDGE_FEATURE_DEGREE ? 0u : id + 1u;
}

// lane 0 only: the share of <w, f> that comes from the topological features
__device__ __forceinline__ float metrics_dot(const MethodList &m, const float *w, const float (&values)[6]) {
    float total = 0.f;
    for (uint32_t k = 0; k < m.n_metrics; ++k) {
        const uint32_t slot = metric_slot(m.metric_id[k]);
        total = fmaf(w[m.metric_offset[k]], values[slot], total);
        if (m.metric_id[k] == B2E_EDGE_FEATURE_DEGREE) total = fmaf(w[m.metric_offset[k] + 1], values[1], total);
    }
    return total;
}

__device__ __forceinline__ bool needs_scalars(const MethodList &m) {
    for (uint32_t k = 0; k < m.n; ++k)
        if (m.id[k] == B2E_EDGE_L2_DISTANCE || m.id[k] == B2E_EDGE_COSINE_SIMILARITY) return true;
    return false;
}

// ---- EdgeTransformer.transform: out[e] = concatenation of the methods ----
__global__ void __launch_bounds__(256) edge_embedding_kernel(const float *__restrict__ features, uint64_t pitch,
                                                             uint32_t dim, const uint32_t *__restrict__ src,
                                                             const uint32_t *__restrict__ dst, uint64_t m,
                                                             MethodList methods, float *__restrict__ out) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t e = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < m; e += warps) {
        const float *a = features + (uint64_t)__ldg(src + e) * pitch;
        const float *b = features + (uint64_t)__ldg(dst + e) * pitch;
        float *row = out + e * methods.size;
        float l2 = 0.f, cosine = 0.f;
        if (needs_scalars(methods)) scalar_features(a, b, dim, lane, l2, cosine);
        for (uint32_t k = 0; k < methods.n; ++k) {
            const uint32_t id = methods.id[k];
            float *o = row + methods.offset[k];
            if (id == B2E_EDGE_L2_DISTANCE) {
                if (lane == 0) o[0] = l2;
            } else if (id == B2E_EDGE_COSINE_SIMILARITY) {
                if (lane == 0) o[0] = cosine;
            } else if (id == B2E_EDGE_CONCATENATE) {
                for (uint32_t j = lane; j < dim; j += 32u) { o[j] = __ldg(a + j); o[dim + j] = __ldg(b + j); }
            } else {
                for (uint32_t j = lane; j < dim; j += 32u) o[j] = elementwise(id, __ldg(a + j), __ldg(b + j));
            }
        }
    }
}

// <w, f(a, b)> over the concatenated methods, every lane ends up with the total
__device__ __forceinline__ float forward_dot(const float *__restrict__ a, const float *__restrict__ b, uint32_t dim,
                                             uint32_t lane, const MethodList &methods, const float *w, float l2,
                                             float cosine) {
    float partial = 0.f;
    for (uint32_t k = 0; k < methods.n; ++k) {
        const uint32_t id = methods.id[k];
        const float *wk = w + methods.offset[k];
        if (id == B2E_EDGE_L2_DISTANCE) {
            if (lane == 0) partial = fmaf(wk[0], l2, partial);
        } else if (id == B2E_EDGE_COSINE_SIMILARITY) {
            if (lane == 0) partial = fmaf(wk[0], cosine, partial);
        } else if (id == B2E_EDGE_CONCATENATE) {
            for (uint32_t j = lane; j < dim; j += 32u)
                partial = fmaf(wk[dim + j], __ldg(b + j), fmaf(wk[j], __ldg(a + j), partial));
        } else {
            for (uint32_t j = lane; j < dim; j += 32u)
                partial = fmaf(wk[j], elementwise(id, __ldg(a + j), __ldg(b + j)), partial);
        }
    }
    return warp_sum(partial);
}

__device__ __forceinline__ float sigmoidf(float z) { return 1.0f / (1.0f + __expf(-z)); }

// ---- the topological features of an edge list, materialised (graph.get_*_scores) ----
__global__ void __launch_bounds__(256) edge_metrics_kernel(GraphView g, const uint32_t *__restrict__ src,
                                                           const uint32_t *__restrict__ dst, uint64_t m,
                                                           MethodList methods, float *__restrict__ out) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t e = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < m; e += warps) {
        float values[6];
        edge_metric_values(g, __ldg(src + e), __ldg(dst + e), lane, values);
        if (lane == 0) {
            float *row = out + e * methods.size;
            for (uint32_t k = 0; k < methods.n_metrics; ++k) {
                const uint32_t slot = metric_slot(methods.metric_id[k]);
                row[methods.metric_offset[k]] = values[slot];
                if (methods.metric_id[k] == B2E_EDGE_FEATURE_DEGREE) row[methods.metric_offset[k] + 1] = values[1];
            }
        }
    }
}

// ---- predict_proba ----
__global__ void __launch_bounds__(256) perceptron_predict_kernel(const float *__restrict__ features, uint64_t pitch,
                                                                 uint32_t dim, const uint32_t *__restrict__ src,
                                                                 const uint32_t *__restrict__ dst, uint64_t m,
                                                                 MethodList methods, GraphView graph,
                                                                 const float *__restrict__ params,
                                                                 float *__restrict__ scores) {
    extern __shared__ float w[];  // size weights + bias
    for (uint32_t j = threadIdx.x; j <= methods.size; j += blockDim.x) w[j] = params[j];
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t e = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < m; e += warps) {
        const float *a = features + (uint64_t)__ldg(src + e) * pitch;
        const float *b = features + (uint64_t)__ldg(dst + e) * pitch;
        float l2 = 0.f, cosine = 0.f;
        if (needs_scalars(methods)) scalar_features(a, b, dim, lane, l2, cosine);
        float z = forward_dot(a, b, dim, lane, methods, w, l2, cosine) + w[methods.size];
        if (methods.n_metrics) {
            float values[6];
            edge_metric_values(graph, __ldg(src + e), __ldg(dst + e), lane, values);
            z += metrics_dot(methods, w, values);  // meaningful on lane 0, which writes the score
        }
        if (lane == 0) scores[e] = sigmoidf(z);
    }
}

struct StepParams {
    const float *features;
    uint64_t pitch;
    uint32_t dim;
    const int64_t *indptr;
    const uint32_t *indices;
    const uint32_t *edge_src;  // source of every directed edge (COO view of the CSR)
    uint32_t n;
    uint64_t nnz;
    uint32_t seed_lo, seed_hi, step, batch;
    uint32_t scale_free, avoid_false_negatives;
    float inv_max_degree;
    const float *params;  // size weights + bias
    float *grad;          // size + 1, accumulated with atomics, cleared by the Adam kernel
    double *loss;         // [0] loss sum, [1] valid samples (of the epoch)
};

__device__ __forceinline__ bool is_edge(const StepParams &p, uint32_t u, uint32_t v) {
    int64_t lo = __ldg(p.indptr + u), hi = __ldg(p.indptr + u + 1);
    const int64_t end = hi;
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(p.indices + mid) < v) lo = mid + 1; else hi = mid;
    }
    return lo < end && __ldg(p.indices + lo) == v;
}

// ---- one minibatch: sample, forward, gradient (shared-memory reduction per CTA) ----
__global__ void __launch_bounds__(256) perceptron_step_kernel(const StepParams p, MethodList methods) {
    extern __shared__ float smem[];
    float *w = smem;                         // size + 1
    float *g = smem + methods.size + 1;      // size + 1
    __shared__ uint32_t s_u[8], s_v[8], s_valid[8];
    __shared__ float s_sums[8][3];
    for (uint32_t j = threadIdx.x; j <= methods.size; j += blockDim.x) { w[j] = p.params[j]; g[j] = 0.f; }
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const GraphView graph = {p.indptr, p.indices, p.inv_max_degree};
    float loss = 0.f, valid_count = 0.f;
    // a CTA takes 8 consecutive samples per round, one per warp (CTA-uniform trip count)
    for (uint32_t base = blockIdx.x * 8u; base < p.batch; base += gridDim.x * 8u) {
        const uint32_t k = base + warp;
        const uint4 r = philox4x32_10(p.seed_lo, p.seed_hi, k, p.step, 0u, TAG_EDGE_SAMPLE << 24);
        const bool positive = (k & 1u) == 0u;
        const uint64_t ex = __umul64hi((uint64_t)r.x << 32, p.nnz), ey = __umul64hi((uint64_t)r.y << 32, p.nnz);
        uint32_t u = 0, v = 0;
        bool valid = k < p.batch;
        if (valid) {
            if (positive) {
                u = __ldg(p.edge_src + ex);
                v = __ldg(p.indices + ex);
            } else if (p.scale_free) {
                u = __ldg(p.edge_src + ex);
                v = __ldg(p.indices + ey);
            } else {
                u = __umulhi(r.x, p.n);
                v = __umulhi(r.y, p.n);
            }
            valid = positive || u != v;
            if (valid && !positive && p.avoid_false_negatives) valid = !is_edge(p, u, v);
        }
        float values[6];
        if (methods.n_metrics) {  // CTA-uniform
            if (lane == 0) {
                s_u[warp] = u; s_v[warp] = v; s_valid[warp] = valid ? 1u : 0u;
                s_sums[warp][0] = s_sums[warp][1] = s_sums[warp][2] = 0.f;
            }
            __syncthreads();
            cta_common_neighbours(graph, s_u, s_v, s_valid, 8u, s_sums);
            __syncthreads();
            if (valid) {
                const float du = (float)(uint32_t)(__ldg(p.indptr + u + 1) - __ldg(p.indptr + u));
                const float dv = (float)(uint32_t)(__ldg(p.indptr + v + 1) - __ldg(p.indptr + v));
                finish_metric_values(graph, du, dv, s_sums[warp][0], s_sums[warp][1], s_sums[warp][2], values);
            }
            __syncthreads();  // s_* are rewritten in the next round
        }
        if (!valid) continue;  // warp-uniform; no CTA-wide barrier below this line
        const float *a = p.features + (uint64_t)u * p.pitch;
        const float *b = p.features + (uint64_t)v * p.pitch;
        float l2 = 0.f, cosine = 0.f;
        if (needs_scalars(methods)) scalar_features(a, b, p.dim, lane, l2, cosine);
        float z = forward_dot(a, b, p.dim, lane, methods, w, l2, cosine) + w[methods.size];
        if (methods.n_metrics) z += metrics_dot(methods, w, values);
        const float prob = sigmoidf(z);
        const float delta = (prob - (positive ? 1.0f : 0.0f)) / (float)p.batch;
        if (lane == 0) {
            loss += -__logf((positive ? prob : 1.0f - prob) + 1e-12f);
            valid_count += 1.0f;
            atomicAdd(g + methods.size, delta);
            for (uint32_t m = 0; m < methods.n_metrics; ++m) {
                const uint32_t slot = metric_slot(methods.metric_id[m]);
                atomicAdd(g + methods.metric_offset[m], delta * values[slot]);
                if (methods.metric_id[m] == B2E_EDGE_FEATURE_DEGREE)
                    atomicAdd(g + methods.metric_offset[m] + 1, delta * values[1]);
            }
        }
        for (uint32_t m = 0; m < methods.n; ++m) {
            const uint32_t id = methods.id[m];
            float *gk = g + methods.offset[m];
            if (id == B2E_EDGE_L2_DISTANCE) {
                if (lane == 0) atomicAdd(gk, delta * l2);
            } else if (id == B2E_EDGE_COSINE_SIMILARITY) {
                if (lane == 0) atomicAdd(gk, delta * cosine);
            } else if (id == B2E_EDGE_CONCATENATE) {
                for (uint32_t j = lane; j < p.dim; j += 32u) {
                    atomicAdd(gk + j, delta * __ldg(a + j));
                    atomicAdd(gk + p.dim + j, delta * __ldg(b + j));
                }
            } else {
                for (uint32_t j = lane; j < p.dim; j += 32u)
                    atomicAdd(gk + j, delta * elementwise(id, __ldg(a + j), __ldg(b + j)));
            }
        }
    }
    __syncthreads();
    for (uint32_t j = threadIdx.x; j <= methods.size; j += blockDim.x)
        if (g[j] != 0.f) atomicAdd(p.grad + j, g[j]);
    if (lane == 0 && valid_count > 0.f) {
        atomicAdd(p.loss, (double)loss);
        atomicAdd(p.loss + 1, (double)valid_count);
    }
}

// ---- Adam (bias correction folded into lr_s on the host); clears the gradient ----
__global__ void __launch_bounds__(256) adam_kernel(float *params, float *m, float *v, float *grad, uint32_t count,
                                                   float beta1, float beta2, float lr_s) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const float gj = grad[j];
    grad[j] = 0.f;
    const float mj = __fadd_rn(__fmul_rn(beta1, m[j]), __fmul_rn(__fsub_rn(1.0f, beta1), gj));
    const float vj = __fadd_rn(__fmul_rn(beta2, v[j]), __fmul_rn(__fmul_rn(__fsub_rn(1.0f, beta2), gj), gj));
    m[j] = mj;
    v[j] = vj;
    params[j] = __fsub_rn(params[j], __fdiv_rn(__fmul_rn(lr_s, mj), __fadd_rn(__fsqrt_rn(vj), 1e-8f)));
}

__global__ void __launch_bounds__(256) perceptron_init_kernel(float *params, uint32_t size, uint32_t seed_lo,
                                                              uint32_t seed_hi) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j > size) return;
    if (j == size) { params[j] = 0.f; return; }
    const uint4 r = philox4x32_10(seed_lo, seed_hi, j, 0u, 0u, TAG_PERCEPTRON_INIT << 24);
    const float u01 = __fmul_rn((float)(r.x >> 8), 5.9604644775390625e-8f);
    const float scale = __fdiv_rn(2.0f, __fsqrt_rn((float)size));
    params[j] = __fmul_rn(__fsub_rn(u01, 0.5f), scale);
}

__global__ void __launch_bounds__(256) edge_sources_kernel(const int64_t *__restrict__ indptr, uint64_t n,
                                                           uint32_t *__restrict__ edge_src) {
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    for (uint64_t v = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < n; v += warps)
        for (int64_t e = __ldg(indptr + v) + lane, end = __ldg(indptr + v + 1); e < end; e += 32) edge_src[e] = (uint32_t)v;
}

}  // namespace b2e

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
using namespace b2e;

struct b2e_features {
    int device = 0;
    DeviceBuffer<float> owned;  // the table of b2e_features_create; empty for a view of a handle's table
    const float *d = nullptr;
    uint64_t n = 0, pitch = 0;
    uint32_t dim = 0;
};

static int build_methods(const uint32_t *ids, uint32_t count, uint32_t dim, const uint32_t *metrics,
                         uint32_t n_metrics, MethodList &out) {
    if (count > MAX_METHODS || n_metrics > MAX_METRICS || (count && !ids) || (n_metrics && !metrics))
        return fail(B2E_ERR_INVALID, "at most 12 edge embedding methods and 5 edge features");
    if (count + n_metrics == 0)
        return fail(B2E_ERR_INVALID, "at least one edge embedding method or edge feature is required");
    out.n = count;
    out.n_metrics = n_metrics;
    out.size = 0;
    for (uint32_t k = 0; k < count; ++k) {
        if (ids[k] > B2E_EDGE_COSINE_SIMILARITY) return fail(B2E_ERR_INVALID, "unknown edge embedding method");
        out.id[k] = ids[k];
        out.offset[k] = out.size;
        out.size += method_width(ids[k], dim);
    }
    for (uint32_t k = 0; k < n_metrics; ++k) {
        if (metrics[k] > B2E_EDGE_FEATURE_PREFERENTIAL_ATTACHMENT)
            return fail(B2E_ERR_INVALID, "unknown edge feature");
        out.metric_id[k] = metrics[k];
        out.metric_offset[k] = out.size;
        out.size += metrics[k] == B2E_EDGE_FEATURE_DEGREE ? 2u : 1u;
    }
    if ((out.size + 1) * 2 * sizeof(float) > 200 * 1024)
        return fail(B2E_ERR_INVALID, "edge embedding too wide for the perceptron kernels");
    return B2E_OK;
}

// every upload holds at least 16 bytes
template <typename T> static cudaError_t alloc(DeviceBuffer<T> &buffer, size_t bytes) {
    return buffer.reserve(std::max<size_t>(bytes, 16));
}

// the support graph of the topological features, uploaded for the duration of a call
// ids in range and rows strictly ascending (walk_kernels.cu: csr_check_kernel): the common-neighbour
// pass and the samplers index and gallop through these arrays without looking again
static int check_csr_contents(const int64_t *h_indptr, const int64_t *d_indptr, const uint32_t *d_indices,
                              uint64_t n) {
    for (uint64_t v = 0; v < n; ++v)
        if (h_indptr[v + 1] < h_indptr[v]) return fail(B2E_ERR_INVALID, "indptr must be non-decreasing");
    DeviceBuffer<int> d_flags;
    int flags = 0;
    CUDA_TRY(d_flags.reserve(sizeof(int)));
    CUDA_TRY(cudaMemset(d_flags.get(), 0, sizeof(int)));
    CUDA_TRY(launch_csr_check(d_indptr, d_indices, n, d_flags.get(), 148, 0));
    CUDA_TRY(cudaMemcpy(&flags, d_flags.get(), sizeof(int), cudaMemcpyDeviceToHost));
    if (flags & 1) return fail(B2E_ERR_INVALID, "a destination node id is out of range");
    if (flags & 2)
        return fail(B2E_ERR_INVALID, "neighbour lists must be sorted strictly ascending within each row");
    return B2E_OK;
}

struct DeviceGraph {
    DeviceBuffer<int64_t> indptr;
    DeviceBuffer<uint32_t> indices;
    GraphView view = {nullptr, nullptr, 0.f};
    int upload(const int64_t *h_indptr, const uint32_t *h_indices, uint64_t n, uint64_t nnz) {
        if (!h_indptr || (!h_indices && nnz) || h_indptr[0] != 0 || (uint64_t)h_indptr[n] != nnz)
            return fail(B2E_ERR_INVALID, "the edge features need the support graph's CSR");
        int64_t max_degree = 1;
        for (uint64_t v = 0; v < n; ++v) max_degree = std::max(max_degree, h_indptr[v + 1] - h_indptr[v]);
        CUDA_TRY(alloc(indptr, (n + 1) * sizeof(int64_t)));
        CUDA_TRY(alloc(indices, nnz * sizeof(uint32_t)));
        CUDA_TRY(cudaMemcpy(indptr.get(), h_indptr, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(indices.get(), h_indices, nnz * sizeof(uint32_t), cudaMemcpyHostToDevice));
        if (int rc = check_csr_contents(h_indptr, indptr.get(), indices.get(), n)) return rc;
        view.indptr = indptr.get();
        view.indices = indices.get();
        view.inv_max_degree = 1.0f / (float)max_degree;
        return B2E_OK;
    }
};

static int use_features_device(const b2e_features *f) {
    if (f) CUDA_TRY(cudaSetDevice(f->device));
    return B2E_OK;
}

extern "C" int b2e_features_create(int device, const float *host, uint64_t n, uint32_t dim, b2e_features **out) {
    if (!host || !out || n == 0 || dim == 0) return fail(B2E_ERR_INVALID, "null or empty node features");
    if (int rc = select_device(device)) return rc;
    std::unique_ptr<b2e_features> f(new b2e_features());
    f->device = device;
    f->n = n;
    f->dim = dim;
    f->pitch = dim;
    CUDA_TRY(f->owned.reserve(n * (uint64_t)dim * sizeof(float)));
    CUDA_TRY(cudaMemcpy(f->owned.get(), host, n * (uint64_t)dim * sizeof(float), cudaMemcpyHostToDevice));
    f->d = f->owned.get();
    *out = f.release();
    return B2E_OK;
}

extern "C" int b2e_features_from_handle(b2e_handle *h, int table, b2e_features **out) {
    if (!h || !out || table < 0 || table > 1) return fail(B2E_ERR_INVALID, "bad argument");
    if (!h->graph.t0.get()) return fail(B2E_ERR_STATE, "the handle holds no tables yet");
    if (int rc = b2e_sync(h)) return rc;
    b2e_features *f = new b2e_features();
    f->device = h->cfg.device;
    f->d = table ? h->graph.t1.get() : h->graph.t0.get();
    f->n = h->n;
    f->dim = h->cfg.embedding_size;
    f->pitch = h->row_stride;
    // a view: valid while the handle lives and keeps its graph
    *out = f;
    return B2E_OK;
}

extern "C" void b2e_features_destroy(b2e_features *f) {
    if (!f) return;
    if (f->owned.get()) cudaSetDevice(f->device);
    delete f;
}

extern "C" int b2e_edge_embedding_size(uint32_t dim, const uint32_t *methods, uint32_t n_methods,
                                       const uint32_t *edge_features, uint32_t n_edge_features, uint32_t *size) {
    MethodList list;
    if (!size) return fail(B2E_ERR_INVALID, "null argument");
    if (int rc = build_methods(methods, n_methods, dim, edge_features, n_edge_features, list)) return rc;
    *size = list.size;
    return B2E_OK;
}

static int upload_edges(uint64_t n, const uint32_t *src, const uint32_t *dst, uint64_t m,
                        DeviceBuffer<uint32_t> &d_src, DeviceBuffer<uint32_t> &d_dst) {
    for (uint64_t e = 0; e < m; ++e)
        if (src[e] >= n || dst[e] >= n) return fail(B2E_ERR_INVALID, "a node id is out of range");
    CUDA_TRY(alloc(d_src, m * sizeof(uint32_t)));
    CUDA_TRY(alloc(d_dst, m * sizeof(uint32_t)));
    CUDA_TRY(cudaMemcpy(d_src.get(), src, m * sizeof(uint32_t), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_dst.get(), dst, m * sizeof(uint32_t), cudaMemcpyHostToDevice));
    return B2E_OK;
}

static unsigned warp_grid(uint64_t warps_wanted) {
    return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((warps_wanted + 7) / 8, 148ull * 8));
}

extern "C" int b2e_edge_embedding(const b2e_features *f, const uint32_t *src, const uint32_t *dst, uint64_t m,
                                  const uint32_t *methods, uint32_t n_methods, float *out) {
    if (!f || (m && (!src || !dst || !out))) return fail(B2E_ERR_INVALID, "null argument");
    MethodList list;
    if (n_methods == 0) return fail(B2E_ERR_INVALID, "at least one edge embedding method is required");
    if (int rc = build_methods(methods, n_methods, f->dim, nullptr, 0, list)) return rc;
    if (m == 0) return B2E_OK;
    CUDA_TRY(cudaSetDevice(f->device));
    DeviceBuffer<uint32_t> d_src, d_dst;
    DeviceBuffer<float> d_out;
    if (int rc = upload_edges(f->n, src, dst, m, d_src, d_dst)) return rc;
    // the materialised embedding is produced in slabs so that it never needs more than 1 GiB
    const uint64_t slab = std::max<uint64_t>(1, (1ull << 28) / list.size);
    CUDA_TRY(alloc(d_out, std::min(slab, m) * list.size * sizeof(float)));
    for (uint64_t done = 0; done < m; done += slab) {
        const uint64_t count = std::min(slab, m - done);
        edge_embedding_kernel<<<warp_grid(count), 256>>>(f->d, f->pitch, f->dim, d_src.get() + done,
                                                        d_dst.get() + done, count, list, d_out.get());
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpy(out + done * list.size, d_out.get(), count * list.size * sizeof(float), cudaMemcpyDeviceToHost));
    }
    return B2E_OK;
}

extern "C" int b2e_edge_metrics(int device, const int64_t *indptr, const uint32_t *indices, uint64_t n, uint64_t nnz,
                                const uint32_t *src, const uint32_t *dst, uint64_t m, const uint32_t *edge_features,
                                uint32_t n_edge_features, float *out) {
    if (m && (!src || !dst || !out)) return fail(B2E_ERR_INVALID, "null argument");
    MethodList list;
    if (n_edge_features == 0) return fail(B2E_ERR_INVALID, "at least one edge feature is required");
    if (int rc = build_methods(nullptr, 0, 0, edge_features, n_edge_features, list)) return rc;
    if (m == 0) return B2E_OK;
    CUDA_TRY(cudaSetDevice(device));
    DeviceGraph graph;
    if (int rc = graph.upload(indptr, indices, n, nnz)) return rc;
    DeviceBuffer<uint32_t> d_src, d_dst;
    DeviceBuffer<float> d_out;
    if (int rc = upload_edges(n, src, dst, m, d_src, d_dst)) return rc;
    CUDA_TRY(alloc(d_out, m * list.size * sizeof(float)));
    edge_metrics_kernel<<<warp_grid(m), 256>>>(graph.view, d_src.get(), d_dst.get(), m, list,
                                               d_out.get());
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(out, d_out.get(), m * list.size * sizeof(float), cudaMemcpyDeviceToHost));
    return B2E_OK;
}

extern "C" int b2e_perceptron_predict(const b2e_features *f, const int64_t *indptr, const uint32_t *indices,
                                      uint64_t n, uint64_t nnz, const uint32_t *src, const uint32_t *dst, uint64_t m,
                                      const uint32_t *methods, uint32_t n_methods, const uint32_t *edge_features,
                                      uint32_t n_edge_features, const float *params, float *scores) {
    if (!params || (m && (!src || !dst || !scores))) return fail(B2E_ERR_INVALID, "null argument");
    if (n_methods && !f) return fail(B2E_ERR_INVALID, "edge embeddings need node features");
    if (f && n_edge_features && n != f->n)
        return fail(B2E_ERR_INVALID, "the graph and the node features disagree on the number of nodes");
    MethodList list;
    if (int rc = build_methods(methods, n_methods, f ? f->dim : 0, edge_features, n_edge_features, list)) return rc;
    if (m == 0) return B2E_OK;
    if (int rc = use_features_device(f)) return rc;
    DeviceGraph graph;
    if (n_edge_features)
        if (int rc = graph.upload(indptr, indices, n, nnz)) return rc;
    DeviceBuffer<uint32_t> d_src, d_dst;
    DeviceBuffer<float> d_params, d_scores;
    if (int rc = upload_edges(f ? f->n : n, src, dst, m, d_src, d_dst)) return rc;
    CUDA_TRY(alloc(d_params, (list.size + 1) * sizeof(float)));
    CUDA_TRY(alloc(d_scores, m * sizeof(float)));
    CUDA_TRY(cudaMemcpy(d_params.get(), params, (list.size + 1) * sizeof(float), cudaMemcpyHostToDevice));
    const size_t smem = (list.size + 1) * sizeof(float);
    CUDA_TRY(cudaFuncSetAttribute(perceptron_predict_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    perceptron_predict_kernel<<<warp_grid(m), 256, smem>>>(f ? f->d : nullptr, f ? f->pitch : 0, f ? f->dim : 0,
                                                           d_src.get(), d_dst.get(), m, list,
                                                           graph.view, d_params.get(), d_scores.get());
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(scores, d_scores.get(), m * sizeof(float), cudaMemcpyDeviceToHost));
    return B2E_OK;
}

extern "C" int b2e_perceptron_fit(const b2e_features *f, const int64_t *indptr, const uint32_t *indices, uint64_t n,
                                  uint64_t nnz, const b2e_perceptron_config *cfg, uint64_t seed, float *params_out,
                                  float *epoch_loss) {
    if (!indptr || !indices || !cfg || !params_out) return fail(B2E_ERR_INVALID, "null argument");
    if (cfg->struct_size != sizeof(b2e_perceptron_config))
        return fail(B2E_ERR_INVALID, "b2e_perceptron_config size mismatch (ABI)");
    if (cfg->n_methods && !f) return fail(B2E_ERR_INVALID, "edge embeddings need node features");
    if (f && n != f->n) return fail(B2E_ERR_INVALID, "the graph and the node features disagree on the number of nodes");
    if (nnz == 0 || indptr[0] != 0 || (uint64_t)indptr[n] != nnz)
        return fail(B2E_ERR_INVALID, "the graph has no edges");
    if (cfg->number_of_edges_per_mini_batch == 0) return fail(B2E_ERR_INVALID, "empty mini-batch");
    if (!(cfg->first_order_decay_factor >= 0.f && cfg->first_order_decay_factor < 1.f) ||
        !(cfg->second_order_decay_factor >= 0.f && cfg->second_order_decay_factor < 1.f))
        return fail(B2E_ERR_INVALID, "decay factors must be in [0, 1)");
    MethodList list;
    if (int rc = build_methods(cfg->methods, cfg->n_methods, f ? f->dim : 0, cfg->edge_features,
                               cfg->n_edge_features, list))
        return rc;
    if (int rc = use_features_device(f)) return rc;
    int64_t max_degree = 1;
    for (uint64_t v = 0; v < n; ++v) max_degree = std::max(max_degree, indptr[v + 1] - indptr[v]);
    const uint32_t count = list.size + 1;
    DeviceBuffer<int64_t> d_indptr;
    DeviceBuffer<uint32_t> d_indices, d_edge_src;
    DeviceBuffer<float> d_params, d_m, d_v, d_grad;
    DeviceBuffer<double> d_loss;
    CUDA_TRY(alloc(d_indptr, (n + 1) * sizeof(int64_t)));
    CUDA_TRY(alloc(d_indices, nnz * sizeof(uint32_t)));
    CUDA_TRY(alloc(d_edge_src, nnz * sizeof(uint32_t)));
    CUDA_TRY(alloc(d_params, count * sizeof(float)));
    CUDA_TRY(alloc(d_m, count * sizeof(float)));
    CUDA_TRY(alloc(d_v, count * sizeof(float)));
    CUDA_TRY(alloc(d_grad, count * sizeof(float)));
    CUDA_TRY(alloc(d_loss, 2 * sizeof(double)));
    CUDA_TRY(cudaMemcpy(d_indptr.get(), indptr, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_indices.get(), indices, nnz * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (int rc = check_csr_contents(indptr, d_indptr.get(), d_indices.get(), n)) return rc;
    CUDA_TRY(cudaMemset(d_m.get(), 0, count * sizeof(float)));
    CUDA_TRY(cudaMemset(d_v.get(), 0, count * sizeof(float)));
    CUDA_TRY(cudaMemset(d_grad.get(), 0, count * sizeof(float)));
    edge_sources_kernel<<<warp_grid(n), 256>>>(d_indptr.get(), n, d_edge_src.get());
    perceptron_init_kernel<<<(count + 255) / 256, 256>>>(d_params.get(), list.size, (uint32_t)seed,
                                                         (uint32_t)(seed >> 32));
    CUDA_TRY(cudaGetLastError());

    StepParams p;
    p.features = f ? f->d : nullptr;
    p.pitch = f ? f->pitch : 0;
    p.dim = f ? f->dim : 0;
    p.inv_max_degree = 1.0f / (float)max_degree;
    p.indptr = d_indptr.get();
    p.indices = d_indices.get();
    p.edge_src = d_edge_src.get();
    p.n = (uint32_t)n;
    p.nnz = nnz;
    p.seed_lo = (uint32_t)seed;
    p.seed_hi = (uint32_t)(seed >> 32);
    p.batch = cfg->number_of_edges_per_mini_batch;
    p.scale_free = cfg->use_scale_free_distribution ? 1u : 0u;
    p.avoid_false_negatives = cfg->avoid_false_negatives ? 1u : 0u;
    p.params = d_params.get();
    p.grad = d_grad.get();
    p.loss = d_loss.get();
    const size_t smem = 2 * (size_t)count * sizeof(float);
    CUDA_TRY(cudaFuncSetAttribute(perceptron_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    const uint64_t steps_per_epoch = std::max<uint64_t>(1, nnz / p.batch);
    const double beta1 = cfg->first_order_decay_factor, beta2 = cfg->second_order_decay_factor;
    uint64_t step = 0;
    for (uint32_t epoch = 0; epoch < cfg->number_of_epochs; ++epoch) {
        CUDA_TRY(cudaMemsetAsync(d_loss.get(), 0, 2 * sizeof(double)));
        for (uint64_t s = 0; s < steps_per_epoch; ++s) {
            ++step;
            p.step = (uint32_t)step;
            perceptron_step_kernel<<<warp_grid(p.batch), 256, smem>>>(p, list);
            const float lr_s = (float)((double)cfg->learning_rate * std::sqrt(1.0 - std::pow(beta2, (double)step)) /
                                       (1.0 - std::pow(beta1, (double)step)));
            adam_kernel<<<(count + 255) / 256, 256>>>(d_params.get(), d_m.get(), d_v.get(),
                                                      d_grad.get(), count, (float)beta1, (float)beta2, lr_s);
        }
        CUDA_TRY(cudaGetLastError());
        if (epoch_loss) {
            double host[2];
            CUDA_TRY(cudaMemcpy(host, d_loss.get(), sizeof(host), cudaMemcpyDeviceToHost));
            epoch_loss[epoch] = host[1] > 0 ? (float)(host[0] / host[1]) : 0.f;
        }
    }
    CUDA_TRY(cudaMemcpy(params_out, d_params.get(), count * sizeof(float), cudaMemcpyDeviceToHost));
    return B2E_OK;
}
