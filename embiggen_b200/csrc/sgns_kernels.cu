// K4 / K5: fused window + negative-sampling SkipGram and CBOW SGD kernels for sm_100a.
//
// Replaces the training half of `ensmallen.models.SkipGram/CBOW.fit_transform`
// (/root/reference/embiggen/embedders/ensmallen_embedders/node2vec.py:99; kwargs
// .../node2vec_skipgram.py:37-119).  One warp per walk, fetched dynamically.  The bound is
// HBM: every (centre, context) pair gathers and scatters K+1 rows of the contextual table
// (2 * 4D bytes each), K of them at random.  The kernel is therefore organised as a software
// pipeline over the *draw sites* of a walk (a pair for SkipGram, a centre for CBOW):
//
//   site s+2 : Philox draw + alias-table gather issued (the ids depend on (seed, walk, site)
//              only, never on the tables, so they can run arbitrarily far ahead);
//   site s+1 : ids resolved, its K+1 target rows prefetched into L2 (CCTL.PF2, one line per
//              lane) so the DRAM latency is paid while site s computes;
//   site s   : rows gathered with 128-bit loads issued back to back (L2 hits), warp-shuffle
//              dot products, sigmoid, axpy, rows scattered back with 128-bit stores
//              (Hogwild: plain stores, no locks).
//
// Floating point follows the normative spec (DESIGN.md): explicit round-to-nearest
// intrinsics, a fixed reduction order and a polynomial sigmoid, so a single-warp launch
// (cfg.deterministic) reproduces the CPU oracle's tables bit for bit.  Prefetches never
// change a value, so both launches run the same code.
#include <algorithm>

#include "sgns_device.cuh"

namespace b2e {

// ---- negative draws: issued one site early, resolved when the alias entry has arrived ----
struct Draw {
    uint32_t idx;  // uniform proposal of this lane (lane < K)
    uint32_t ry;   // second random word, compared with the alias threshold
    uint2 entry;   // {threshold, alias} gathered from the alias table (in flight)
};

__device__ __forceinline__ Draw draw_issue(const TrainParams &p, uint32_t wid_lo, uint32_t wid_hi,
                                           uint32_t site, uint32_t lane) {
    Draw d;
    d.idx = PAD;
    d.ry = 0;
    d.entry = make_uint2(0xFFFFFFFFu, 0u);
    if (lane < p.negatives) {
        const uint4 r = philox4x32_10(p.seed_lo, p.seed_hi, wid_lo, wid_hi, site,
                                      (TAG_NEG << 24) | lane);
        d.idx = __umulhi(r.x, p.n);
        d.ry = r.y;
        if (p.use_alias) d.entry = __ldg(p.alias + d.idx);
    }
    return d;
}

// Returns the target mask of the site: bit 0 = positive, bit k+1 = negative k is valid.  A draw
// equal to the centre, the context or an earlier draw of the same site is dropped.
__device__ __forceinline__ uint32_t draw_resolve(const TrainParams &p, const Draw &d, uint32_t lane,
                                                 uint32_t centre, uint32_t context, uint32_t &neg) {
    neg = d.idx;
    if (p.use_alias && lane < p.negatives) neg = d.ry < d.entry.x ? d.idx : d.entry.y;
    const uint32_t same = __match_any_sync(FULL, neg);
    const bool valid = lane < p.negatives && neg != centre && neg != context &&
                       (same & ((1u << lane) - 1u)) == 0u;
    return (__ballot_sync(FULL, valid) << 1) | 1u;
}

// One L2 prefetch per 128 B line of every row the next site will touch: slot 0 = row `first`
// of T1, slots 1..K = the valid negatives (T1), slot K+1 = row `extra` of T0 (PAD: none).
__device__ __forceinline__ void prefetch_site(const TrainParams &p, uint32_t lane, uint32_t first,
                                              uint32_t neg, uint32_t vmask, uint32_t extra) {
    const uint32_t row_bytes = p.chunks * 16u;
    const uint32_t slots = p.negatives + 2u;
    for (uint32_t first_t = 0; first_t < slots * 5u; first_t += 32u) {  // warp-uniform trip count
        const uint32_t t = first_t + lane;
        const uint32_t slot = t / 5u, line = t - slot * 5u;
        const uint32_t id_neg = __shfl_sync(FULL, neg, (slot - 1u) & 31u);
        const uint32_t id = slot == 0 ? first : (slot <= p.negatives ? id_neg : extra);
        bool on = slot < slots;
        if (on) on = slot <= p.negatives ? ((vmask >> slot) & 1u) : (extra != PAD);
        if (on) {
            const float *base = (slot <= p.negatives ? p.t1 : p.t0) + (uint64_t)id * p.row_stride;
            const uint32_t head = (uint32_t)(reinterpret_cast<uintptr_t>(base) & 127u);
            if (line * 128u < head + row_bytes) {
                const char *addr = reinterpret_cast<const char *>(base) - head + line * 128u;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(addr));
            }
        }
    }
}

// Score h against slot 0 (= positive) and the valid negatives, in batches of NT rows whose
// loads are all issued before the first use; acc += sum g * row (pre-update rows).
template <int CH, int NT>
__device__ __forceinline__ void apply_targets(const TrainParams &p, uint32_t chunks, uint32_t lane,
                                              const float4 (&h)[CH], float lr, uint32_t positive,
                                              uint32_t neg, uint32_t vmask, float4 (&acc)[CH],
                                              float &loss_acc, unsigned long long &n_targets) {
    const uint32_t K = p.negatives;
    for (uint32_t b = 0; b <= K; b += NT) {
        float4 rows[NT][CH];
        uint32_t ids[NT];
#pragma unroll
        for (int s = 0; s < NT; ++s) {
            const uint32_t slot = b + s;
            const uint32_t id = slot == 0 ? positive : __shfl_sync(FULL, neg, (slot - 1) & 31u);
            const bool on = slot <= K && ((vmask >> slot) & 1u);
            ids[s] = on ? id : PAD;
            if (on) load_row<CH>(p.t1 + (uint64_t)id * p.row_stride, chunks, lane, rows[s]);
        }
        float my_f = 0.0f;
        bool my_on = false;
#pragma unroll
        for (int s = 0; s < NT; ++s) {
            if (ids[s] != PAD) {
                float f = warp_dot<CH>(h, rows[s]);
                if (p.scale_dot) f = __fmul_rn(f, p.inv_scale);
                if (lane == (uint32_t)s) { my_f = f; my_on = true; }
            }
        }
        float g_mine = 0.0f;
        bool apply = false;
        if (my_on && !(fabsf(my_f) > p.clip)) {
            const bool is_positive = (b + lane) == 0;
            const float e = exp_det(-my_f);
            const float sigmoid = __fdiv_rn(1.0f, __fadd_rn(1.0f, e));
            g_mine = __fmul_rn(__fsub_rn(is_positive ? 1.0f : 0.0f, sigmoid), lr);
            // -log sigmoid(f) = log(1 + e^-f);  -log sigmoid(-f) = log(1 + e^-f) + f
            loss_acc += __logf(1.0f + e) + (is_positive ? 0.0f : my_f);
            apply = true;
        }
        const uint32_t amask = __ballot_sync(FULL, apply);
        n_targets += __popc(__ballot_sync(FULL, my_on));
#pragma unroll
        for (int s = 0; s < NT; ++s) {
            if ((amask >> s) & 1u) {
                const float g = __shfl_sync(FULL, g_mine, s);
#pragma unroll
                for (int ch = 0; ch < CH; ++ch) {
                    const float4 old = rows[s][ch];
                    acc[ch].x = __fmaf_rn(g, old.x, acc[ch].x);
                    acc[ch].y = __fmaf_rn(g, old.y, acc[ch].y);
                    acc[ch].z = __fmaf_rn(g, old.z, acc[ch].z);
                    acc[ch].w = __fmaf_rn(g, old.w, acc[ch].w);
                    rows[s][ch].x = __fmaf_rn(g, h[ch].x, old.x);
                    rows[s][ch].y = __fmaf_rn(g, h[ch].y, old.y);
                    rows[s][ch].z = __fmaf_rn(g, h[ch].z, old.z);
                    rows[s][ch].w = __fmaf_rn(g, h[ch].w, old.w);
                }
                store_row<CH>(p.t1 + (uint64_t)ids[s] * p.row_stride, chunks, lane, rows[s]);
            }
        }
    }
}

template <int CH, int NT>
__device__ __forceinline__ void skipgram_walk(const TrainParams &p, const uint32_t *walk, uint64_t wid,
                                              uint32_t lane, float &loss_acc,
                                              unsigned long long &n_pairs,
                                              unsigned long long &n_targets) {
    const uint32_t chunks = p.chunks;
    const uint32_t L = p.walk_length, W = p.window;
    const uint32_t wid_lo = (uint32_t)wid, wid_hi = (uint32_t)(wid >> 32);

    PairCursor scan;
    scan.i = 0xFFFFFFFFu; scan.j = 0; scan.c = PAD; scan.o = PAD; scan.hi = 0;
    bool ok_cur = next_pair(p, wid_lo, wid_hi, walk, L, W, scan);
    if (!ok_cur) return;
    PairCursor cur = scan;
    uint32_t neg_cur;
    uint32_t vmask_cur;
    {
        const Draw d = draw_issue(p, wid_lo, wid_hi, (cur.i << 16) | cur.j, lane);
        vmask_cur = draw_resolve(p, d, lane, cur.c, cur.o, neg_cur);
    }
    bool ok_nxt = next_pair(p, wid_lo, wid_hi, walk, L, W, scan);
    PairCursor nxt = scan;
    Draw draw_nxt = draw_issue(p, wid_lo, wid_hi, (nxt.i << 16) | nxt.j, lane);

    float4 h[CH], acc[CH];
    uint32_t loaded = 0xFFFFFFFFu;  // position of the centre whose row is in h
    float lr = p.lr;
    while (ok_cur) {
        // site s+1: ids are here by now; prefetch its rows into L2
        uint32_t neg_nxt = PAD, vmask_nxt = 0;
        if (ok_nxt) {
            vmask_nxt = draw_resolve(p, draw_nxt, lane, nxt.c, nxt.o, neg_nxt);
            prefetch_site(p, lane, nxt.o, neg_nxt, vmask_nxt, nxt.i != cur.i ? nxt.c : PAD);
        }
        // site s+2: start its draw
        const bool ok_far = ok_nxt && next_pair(p, wid_lo, wid_hi, walk, L, W, scan);
        const PairCursor far = scan;
        Draw draw_far = draw_nxt;
        if (ok_far) draw_far = draw_issue(p, wid_lo, wid_hi, (far.i << 16) | far.j, lane);

        // site s: train the pair
        float *crow = p.t0 + (uint64_t)cur.c * p.row_stride;
        if (loaded != cur.i) {
            load_row<CH>(crow, chunks, lane, h);
            lr = centre_lr(p, cur.c);
            loaded = cur.i;
        }
        zero_rows<CH>(acc);
        apply_targets<CH, NT>(p, chunks, lane, h, lr, cur.o, neg_cur, vmask_cur, acc, loss_acc,
                              n_targets);
        add_rows<CH>(h, acc);
        ++n_pairs;
        if (!ok_nxt || nxt.i != cur.i) store_row<CH>(crow, chunks, lane, h);

        cur = nxt; neg_cur = neg_nxt; vmask_cur = vmask_nxt; ok_cur = ok_nxt;
        nxt = far; draw_nxt = draw_far; ok_nxt = ok_far;
    }
}

template <int CH, int NT>
__device__ __forceinline__ void cbow_walk(const TrainParams &p, const uint32_t *walk, uint64_t wid,
                                          uint32_t lane, float &loss_acc, unsigned long long &n_pairs,
                                          unsigned long long &n_targets) {
    const uint32_t chunks = p.chunks;
    const uint32_t L = p.walk_length, W = p.window;
    const uint32_t wid_lo = (uint32_t)wid, wid_hi = (uint32_t)(wid >> 32);

    uint32_t c_cur = PAD, c_nxt = PAD, c_far = PAD;
    uint32_t i_cur = next_centre(p, wid_lo, wid_hi, walk, L, W, 0, c_cur);
    if (i_cur >= L) return;
    uint32_t neg_cur, vmask_cur;
    {
        const Draw d = draw_issue(p, wid_lo, wid_hi, (i_cur << 16) | 0xFFFFu, lane);
        vmask_cur = draw_resolve(p, d, lane, c_cur, c_cur, neg_cur);
    }
    uint32_t i_nxt = next_centre(p, wid_lo, wid_hi, walk, L, W, i_cur + 1, c_nxt);
    Draw draw_nxt = draw_issue(p, wid_lo, wid_hi, (i_nxt << 16) | 0xFFFFu, lane);

    while (i_cur < L) {
        uint32_t neg_nxt = PAD, vmask_nxt = 0;
        if (i_nxt < L) {
            vmask_nxt = draw_resolve(p, draw_nxt, lane, c_nxt, c_nxt, neg_nxt);
            // the context rows of the next centre are this centre's neighbours (hot) except the
            // one entering the window
            const uint32_t entering = i_nxt + W < L ? __ldg(walk + i_nxt + W) : PAD;
            prefetch_site(p, lane, c_nxt, neg_nxt, vmask_nxt, entering);
        }
        const uint32_t i_far = i_nxt < L ? next_centre(p, wid_lo, wid_hi, walk, L, W, i_nxt + 1, c_far) : L;
        Draw draw_far = draw_nxt;
        if (i_far < L) draw_far = draw_issue(p, wid_lo, wid_hi, (i_far << 16) | 0xFFFFu, lane);

        const uint32_t i = i_cur, c = c_cur;
        const float lr = centre_lr(p, c);
        const uint32_t lo = i > W ? i - W : 0u;
        const uint32_t hi = i + W < L - 1 ? i + W : L - 1;
        float4 h[CH], acc[CH], row[CH];
        uint32_t m = 0;
        for (uint32_t j = lo; j <= hi; ++j) {
            if (j == i) continue;
            const uint32_t o = __ldg(walk + j);
            if (o == PAD || o == c) continue;
            if (m == 0) {
                load_row<CH>(p.t0 + (uint64_t)o * p.row_stride, chunks, lane, h);
            } else {
                load_row<CH>(p.t0 + (uint64_t)o * p.row_stride, chunks, lane, row);
                add_rows<CH>(h, row);
            }
            ++m;
        }
        const float fm = (float)m;
#pragma unroll
        for (int ch = 0; ch < CH; ++ch) {
            h[ch].x = __fdiv_rn(h[ch].x, fm);
            h[ch].y = __fdiv_rn(h[ch].y, fm);
            h[ch].z = __fdiv_rn(h[ch].z, fm);
            h[ch].w = __fdiv_rn(h[ch].w, fm);
        }
        zero_rows<CH>(acc);
        apply_targets<CH, NT>(p, chunks, lane, h, lr, c, neg_cur, vmask_cur, acc, loss_acc,
                              n_targets);
        for (uint32_t j = lo; j <= hi; ++j) {
            if (j == i) continue;
            const uint32_t o = __ldg(walk + j);
            if (o == PAD || o == c) continue;
            float *orow = p.t0 + (uint64_t)o * p.row_stride;
            load_row<CH>(orow, chunks, lane, row);
            add_rows<CH>(row, acc);
            store_row<CH>(orow, chunks, lane, row);
        }
        n_pairs += m;

        i_cur = i_nxt; c_cur = c_nxt; neg_cur = neg_nxt; vmask_cur = vmask_nxt;
        i_nxt = i_far; c_nxt = c_far; draw_nxt = draw_far;
    }
}

template <int MODEL, int CH, int NT, int OCC>
__global__ void __launch_bounds__(256, OCC) train_kernel(const TrainParams p) {
    const uint32_t lane = threadIdx.x & 31u;
    float loss_acc = 0.0f;
    unsigned long long n_pairs = 0, n_targets = 0;
    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(&p.counters->work_counter, 1ull);
        w = __shfl_sync(FULL, w, 0);
        if (w >= p.n_walks) break;
        const uint64_t wid = p.first_walk + w * p.walk_id_stride;
        const uint32_t *walk = p.walks + w * (uint64_t)p.walk_length;
        if (MODEL == B2E_SKIPGRAM)
            skipgram_walk<CH, NT>(p, walk, wid, lane, loss_acc, n_pairs, n_targets);
        else
            cbow_walk<CH, NT>(p, walk, wid, lane, loss_acc, n_pairs, n_targets);
    }
    double loss = (double)loss_acc;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) loss += __shfl_xor_sync(FULL, loss, off);
    if (lane == 0) {
        atomicAdd(&p.counters->pairs, n_pairs);
        atomicAdd(&p.counters->targets, n_targets);
        atomicAdd(&p.counters->loss_sum, loss);
    }
}

template <int MODEL, int CH, int NT, int OCC>
static cudaError_t launch_one(const TrainParams &p, bool deterministic, int sm_count,
                              uint64_t max_warps, cudaStream_t stream) {
    cudaError_t err = cudaMemsetAsync(&p.counters->work_counter, 0, sizeof(unsigned long long), stream);
    if (err != cudaSuccess) return err;
    if (deterministic) {
        train_kernel<MODEL, CH, NT, OCC><<<1, 32, 0, stream>>>(p);
        return cudaGetLastError();
    }
    const int block = 256;
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, train_kernel<MODEL, CH, NT, OCC>,
                                                        block, 0);
    if (err != cudaSuccess) return err;
    if (per_sm < 1) per_sm = 1;
    uint64_t grid = (uint64_t)sm_count * per_sm;  // persistent: every CTA resident, walks fetched
    const uint64_t needed = (std::min<uint64_t>(p.n_walks, max_warps) + 7) / 8;
    if (grid > needed) grid = needed;
    if (grid < 1) grid = 1;
    train_kernel<MODEL, CH, NT, OCC><<<(unsigned)grid, block, 0, stream>>>(p);
    return cudaGetLastError();
}

template <int MODEL>
static cudaError_t launch_model(const TrainParams &p, bool deterministic, int sm_count,
                                uint64_t max_warps, cudaStream_t stream) {
    const uint32_t chunks = p.chunks;
    if (chunks <= 32) {
        if (p.negatives + 1 <= 6) return launch_one<MODEL, 1, 6, 3>(p, deterministic, sm_count, max_warps, stream);
        return launch_one<MODEL, 1, 11, 2>(p, deterministic, sm_count, max_warps, stream);
    }
    if (chunks <= 64) return launch_one<MODEL, 2, 6, 2>(p, deterministic, sm_count, max_warps, stream);
    if (chunks <= 128) return launch_one<MODEL, 4, 3, 2>(p, deterministic, sm_count, max_warps, stream);
    return cudaErrorInvalidValue;
}

cudaError_t launch_train(const TrainParams &p, uint32_t model, bool deterministic, int sm_count,
                         uint64_t max_warps, cudaStream_t stream) {
    if (p.n_walks == 0) return cudaSuccess;
    // production path: shared-memory pipelined kernel; the register path takes the other shapes
    if (model == B2E_SKIPGRAM && p.shared_negatives)  // one kernel, no register-staged twin
        return launch_train_pipe(p, model, deterministic, sm_count, max_warps, stream);
    if (pipe_supported(p, model))
        return launch_train_pipe(p, model, deterministic, sm_count, max_warps, stream);
    if (model == B2E_SKIPGRAM) return launch_model<B2E_SKIPGRAM>(p, deterministic, sm_count, max_warps, stream);
    return launch_model<B2E_CBOW>(p, deterministic, sm_count, max_warps, stream);
}

// ---- table initialisation: one thread per float4 chunk ----
__global__ void __launch_bounds__(256) init_kernel(float *t0, float *t1, uint64_t n,
                                                   uint32_t embedding_size, uint32_t row_stride,
                                                   uint32_t seed_lo, uint32_t seed_hi) {
    const uint32_t chunks = row_stride >> 2;
    const uint64_t total = n * chunks * 2;
    const float dim = (float)embedding_size;
    for (uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t per_table = n * chunks;
        const uint32_t table = idx >= per_table;
        const uint64_t local = table ? idx - per_table : idx;
        const uint64_t row = local / chunks;
        const uint32_t ch = (uint32_t)(local - row * chunks);
        const uint4 r = philox4x32_10(seed_lo, seed_hi, (uint32_t)row, (uint32_t)(row >> 32), ch,
                                      (table ? TAG_INIT1 : TAG_INIT0) << 24);
        const uint32_t words[4] = {r.x, r.y, r.z, r.w};
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float u01 = __fmul_rn((float)(words[e] >> 8), 5.9604644775390625e-8f);
            v[e] = (4u * ch + e) < embedding_size ? __fdiv_rn(__fsub_rn(u01, 0.5f), dim) : 0.0f;
        }
        float *dst = (table ? t1 : t0) + row * row_stride + 4u * ch;
        *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    }
}

cudaError_t launch_init_tables(float *t0, float *t1, uint64_t n, uint32_t embedding_size,
                               uint32_t row_stride, uint64_t seed, cudaStream_t stream) {
    const uint64_t total = n * (row_stride >> 2) * 2;
    uint64_t grid = (total + 255) / 256;
    if (grid > 148ull * 32) grid = 148ull * 32;
    if (grid == 0) return cudaSuccess;
    init_kernel<<<(unsigned)grid, 256, 0, stream>>>(t0, t1, n, embedding_size, row_stride,
                                                    (uint32_t)seed, (uint32_t)(seed >> 32));
    return cudaGetLastError();
}

}  // namespace b2e
