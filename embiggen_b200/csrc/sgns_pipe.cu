// K4 (production path): SkipGram negative-sampling SGD as a per-warp asynchronous pipeline
// staged through shared memory (sm_100a).
//
// Replaces the training half of `ensmallen.models.SkipGram.fit_transform`
// (/root/reference/embiggen/embedders/ensmallen_embedders/node2vec.py:99; kwargs
// .../node2vec_skipgram.py:37-119).  One warp per walk.  The kernel is HBM-latency/-bandwidth
// bound: each (centre, context) pair gathers and scatters K+1 rows of the contextual table, K
// of them at random.  Every gather is therefore an asynchronous global->shared copy
// (cp.async / LDGSTS, no register target, L2-only) issued one pair ahead into a two-stage
// per-warp ring, and the alias-table gathers of the negative draws run two pairs ahead:
//
//   iteration p :  wait(all copies committed in iteration p-1)
//                  resolve the ids of pair p+1 from its alias entries (shared memory)
//                  issue the row copies of pair p+1  -> stage (p+1)&1        } one commit
//                  Philox draw of pair p+2, issue its alias-entry copies     } group
//                  train pair p out of stage p&1: dots (LDS.128 + transposed warp reduction),
//                  sigmoid, axpy, rows scattered to global with 128-bit stores (Hogwild)
//
// The walk itself is staged in shared memory once (its tokens are re-read 2W+1 times each on
// the critical path of the pair cursor).  A row of pair p+1 that pair p is about to update
// (repeated context, a negative equal to a neighbour) would be copied stale; such pairs are
// detected (one MATCH over the two id sets) and their copies are issued after pair p's stores
// instead.  Lane l copies, reads and stores chunk l of every row, so no cross-lane
// shared-memory hazard exists on the rows, and the deterministic single-warp launch
// reproduces the CPU oracle bit for bit: the additions of the transposed reduction are the
// same additions, in the same order, as the oracle's xor-butterfly.
#include <algorithm>

#include "sgns_device.cuh"

namespace b2e {

constexpr int PIPE_SLOTS = 16;  // K + 1 targets at most

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ float4 lds128(const float *smem) {
    return *reinterpret_cast<const float4 *>(smem);
}

// Sum 16 per-lane partials over the 32 lanes.  Level `off` pairs lane l with l^off exactly like
// an xor-butterfly, but each lane keeps only half of the values it holds, so 16 shuffles do the
// work of 80.  Afterwards lane l holds the total of value (l >> 1) & 15.
__device__ __forceinline__ float reduce16(float (&v)[16], uint32_t lane) {
#pragma unroll
    for (int n = 8, off = 16; n >= 1; n >>= 1, off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int k = 0; k < n; ++k) {
            const float send = upper ? v[k] : v[k + n];
            const float keep = upper ? v[k + n] : v[k];
            v[k] = __fadd_rn(keep, __shfl_xor_sync(FULL, send, off));
        }
    }
    return __fadd_rn(v[0], __shfl_xor_sync(FULL, v[0], 1));
}

// stochastic_downsample_by_degree: one bit per walk position, set when the centre there is
// skipped; lane t evaluates position t (one Philox block per position instead of one per lane
// and position), the words live right behind the staged walk
__device__ __forceinline__ void stage_skip_mask(const TrainParams &p, uint32_t wid_lo, uint32_t wid_hi,
                                                uint32_t *walk, uint32_t L, uint32_t lane) {
    if (!p.downsample) return;
    uint32_t *mask = walk + ((L + 31u) & ~31u);
    for (uint32_t base = 0; base < L; base += 32u) {
        const uint32_t t = base + lane;
        bool skip = false;
        if (t < L) {
            const uint32_t c = walk[t];  // written by this very lane just above
            skip = c != PAD && skip_centre(p, wid_lo, wid_hi, t, c);
        }
        const uint32_t word = __ballot_sync(FULL, skip);
        if (lane == 0) mask[base >> 5] = word;
    }
    __syncwarp();
}

// per-warp carve-up of dynamic shared memory; everything exists in two stages
struct PipeSmem {
    float *rows_base;    // [2][K + 2][row_stride]: target rows, then the centre row of T0
    uint2 *alias_base;   // [2][32] alias entries of a draw in flight
    uint32_t *ids_base;  // [2][PIPE_SLOTS] target id per slot (sentinel when the slot is off)
    uint32_t *walk;      // [walk_length rounded up to 32] the warp's current walk
    uint32_t stage_floats, pitch;  // floats per stage / per staged row
    __device__ __forceinline__ float *rows(uint32_t stage) const { return rows_base + stage * stage_floats; }
    __device__ __forceinline__ uint2 *alias(uint32_t a) const { return alias_base + a * 32u; }
    __device__ __forceinline__ uint32_t *ids(uint32_t stage) const { return ids_base + stage * PIPE_SLOTS; }
};

// `chunks` float4 per row are staged (dense pitch in shared memory, 128 B-aligned pitch in HBM)
__host__ __device__ __forceinline__ uint32_t pipe_warp_bytes(uint32_t negatives, uint32_t chunks,
                                                             uint32_t walk_length) {
    return 2u * (negatives + 2u) * chunks * 16u + 2u * 32u * 8u + 2u * PIPE_SLOTS * 4u +
           ((walk_length + 31u) & ~31u) * 4u +              // the walk
           ((((walk_length + 31u) / 32u) * 4u + 15u) & ~15u);  // centre skip mask, slab stays 16 B aligned
}

// what a thread needs to address its 16 B chunk of any row
struct LaneView {
    const char *t0, *t1;  // table bases advanced by 16 * lane bytes
    uint32_t row_bytes;   // 32-bit on purpose: id * row_bytes is then a single widening multiply
    __device__ __forceinline__ const char *row0(uint32_t id) const { return t0 + (uint64_t)id * row_bytes; }
    __device__ __forceinline__ const char *row1(uint32_t id) const { return t1 + (uint64_t)id * row_bytes; }
    uint32_t smem_chunk;  // 4 * min(lane, chunks - 1): lanes past the row re-read its last chunk
    bool active;          // lane < chunks; only active lanes copy and store
};

// ids of the targets of a pair, one per lane: lane 0 = context, lane k+1 = negative k;
// lanes whose slot is off get a sentinel that can never equal a node id or another sentinel
__device__ __forceinline__ uint32_t slot_ids(uint32_t lane, uint32_t context, uint32_t neg,
                                             uint32_t vmask) {
    const uint32_t shifted = __shfl_up_sync(FULL, neg, 1);
    const uint32_t id = lane == 0 ? context : shifted;
    return ((vmask >> lane) & 1u) ? id : (0xFFFFFF00u | lane);
}

// KP1 = K + 1 when known at compile time (0: runtime, up to PIPE_SLOTS); ALL: every slot is on;
// SHARED (skipgram_shared_kernel): the slots are the K negatives alone, KP1 stands for K
template <int KP1, bool ALL, bool SHARED = false>
__device__ __forceinline__ void issue_rows(const TrainParams &p, const PipeSmem &sm, const LaneView &v,
                                           uint32_t stage, uint32_t lane, uint32_t my_id,
                                           uint32_t vmask, uint32_t centre_or_pad) {
    if (lane < PIPE_SLOTS) sm.ids(stage)[lane] = my_id;
    __syncwarp();  // ids are read back by every lane when the pair is trained
    float *dst = sm.rows(stage) + 4u * lane;
    const uint32_t slots = KP1 ? (uint32_t)KP1 : p.negatives + (SHARED ? 0u : 1u);
    constexpr int S = KP1 ? KP1 : PIPE_SLOTS;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        if ((uint32_t)s < slots && (ALL || ((vmask >> s) & 1u))) {
            const uint32_t id = __shfl_sync(FULL, my_id, s);
            if (v.active) cp_async16(dst + (uint32_t)s * sm.pitch, v.row1(id));
        }
    }
    if (centre_or_pad != PAD && v.active)
        cp_async16(dst + slots * sm.pitch, v.row0(centre_or_pad));
}

// dots, sigmoid, axpy and scatter of the targets of one draw site out of stage `stage`;
// returns this lane's chunk of sum g * row (rows as they were before the update)
// SHARED: every slot is a negative that stands for `weight` pairs (skipgram_shared_kernel)
template <int KP1, bool ALL, bool SHARED = false>
__device__ __forceinline__ float4 train_site(const TrainParams &p, const PipeSmem &sm, const LaneView &v,
                                             uint32_t stage, uint32_t lane, uint32_t vmask, float lr,
                                             const float4 &h, float &loss_acc, float weight = 1.0f) {
    // Lanes past the end of the row read its last chunk instead of branching; their h is zero,
    // so they add nothing to a score; their stores are predicated off and their acc is dropped.
    const float *rows = sm.rows(stage) + v.smem_chunk;
    const uint32_t slots = KP1 ? (uint32_t)KP1 : p.negatives + (SHARED ? 0u : 1u);
    constexpr int S = KP1 ? KP1 : PIPE_SLOTS;
    float part[16];
#pragma unroll
    for (int s = 0; s < 16; ++s) {
        float d = 0.0f;
        if (s < S && (uint32_t)s < slots && (ALL || ((vmask >> s) & 1u))) {
            const float4 r = lds128(rows + (uint32_t)s * sm.pitch);
            d = __fmaf_rn(h.x, r.x, d);
            d = __fmaf_rn(h.y, r.y, d);
            d = __fmaf_rn(h.z, r.z, d);
            d = __fmaf_rn(h.w, r.w, d);
        }
        part[s] = d;
    }
    float f = reduce16(part, lane);  // lane l: score of slot (l >> 1) & 15
    if (p.scale_dot) f = __fmul_rn(f, p.inv_scale);
    const uint32_t my_slot = (lane >> 1) & 15u;
    const bool my_on = (vmask >> my_slot) & 1u;  // vmask has no bit above K
    float g_mine = 0.0f;
    bool apply = false;
    if (my_on && !(fabsf(f) > p.clip)) {
        const float e = exp_det(-f);
        const float sigmoid = __fdiv_rn(1.0f, __fadd_rn(1.0f, e));
        // -log sigmoid(f) = log(1 + e^-f);  -log sigmoid(-f) = log(1 + e^-f) + f
        if (SHARED) {
            g_mine = __fmul_rn(__fmul_rn(__fsub_rn(0.0f, sigmoid), lr), weight);
            if ((lane & 1u) == 0) loss_acc += weight * (__logf(1.0f + e) + f);
        } else {
            g_mine = __fmul_rn(__fsub_rn(my_slot == 0 ? 1.0f : 0.0f, sigmoid), lr);
            if ((lane & 1u) == 0) loss_acc += __logf(1.0f + e) + (my_slot == 0 ? 0.0f : f);
        }
        apply = true;
    }
    const uint32_t amask = __ballot_sync(FULL, apply);  // bits 2s, 2s+1: slot s is applied
    constexpr uint32_t all_bits = KP1 >= 16 ? FULL : ((1u << (2 * (KP1 ? KP1 : 1))) - 1u);
    const bool all_applied = KP1 != 0 && ALL && amask == all_bits;
    const uint32_t *ids = sm.ids(stage);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int s = 0; s < S; ++s) {
        if (all_applied || ((amask >> (2 * s)) & 1u)) {
            const float g = __shfl_sync(FULL, g_mine, 2 * s);
            const uint32_t id = ids[s];
            float4 r = lds128(rows + (uint32_t)s * sm.pitch);
            acc.x = __fmaf_rn(g, r.x, acc.x);
            acc.y = __fmaf_rn(g, r.y, acc.y);
            acc.z = __fmaf_rn(g, r.z, acc.z);
            acc.w = __fmaf_rn(g, r.w, acc.w);
            r.x = __fmaf_rn(g, h.x, r.x);
            r.y = __fmaf_rn(g, h.y, r.y);
            r.z = __fmaf_rn(g, h.z, r.z);
            r.w = __fmaf_rn(g, h.w, r.w);
            if (v.active) *reinterpret_cast<float4 *>(const_cast<char *>(v.row1(id))) = r;
        }
    }
    if (!v.active) acc = make_float4(0.f, 0.f, 0.f, 0.f);
    return acc;
}

__device__ __forceinline__ void add4(float4 &a, const float4 &b) {
    a.x = __fadd_rn(a.x, b.x);
    a.y = __fadd_rn(a.y, b.y);
    a.z = __fadd_rn(a.z, b.z);
    a.w = __fadd_rn(a.w, b.w);
}

// MINB: CTAs per SM the register allocation is held to (4: 121 registers; 3 for tables of 32 GiB
// and more, see launch_train_pipe)
template <int KP1, int MINB = 4>
__global__ void __launch_bounds__(128, MINB) skipgram_pipe_kernel(const TrainParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t K = KP1 ? (uint32_t)(KP1 - 1) : p.negatives;
    const uint32_t L = p.walk_length, W = p.window;
    const uint32_t full_mask = (2u << K) - 1u;  // K + 1 ones
    PipeSmem sm;
    {
        unsigned char *base = smem_raw + warp * pipe_warp_bytes(K, p.chunks, L);
        sm.pitch = p.chunks * 4u;
        sm.stage_floats = (K + 2u) * sm.pitch;
        sm.rows_base = reinterpret_cast<float *>(base);
        sm.alias_base = reinterpret_cast<uint2 *>(sm.rows_base + 2u * sm.stage_floats);
        sm.ids_base = reinterpret_cast<uint32_t *>(sm.alias_base + 64);
        sm.walk = sm.ids_base + 2 * PIPE_SLOTS;
    }
    LaneView v;
    v.t0 = reinterpret_cast<const char *>(p.t0) + 16u * lane;
    v.t1 = reinterpret_cast<const char *>(p.t1) + 16u * lane;
    v.row_bytes = p.row_stride * 4u;
    v.active = lane < p.chunks;
    v.smem_chunk = 4u * (lane < p.chunks ? lane : p.chunks - 1u);
    float loss_acc = 0.0f;
    unsigned long long n_pairs = 0, n_targets = 0;

    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(&p.counters->work_counter, 1ull);
        w = __shfl_sync(FULL, w, 0);
        if (w >= p.n_walks) break;
        const uint64_t wid = p.first_walk + w * p.walk_id_stride;
        const uint32_t wid_lo = (uint32_t)wid, wid_hi = (uint32_t)(wid >> 32);
        {
            const uint32_t *src = p.walks + w * (uint64_t)L;
            __syncwarp();
            for (uint32_t t = lane; t < L; t += 32u) sm.walk[t] = __ldg(src + t);
            stage_skip_mask(p, wid_lo, wid_hi, sm.walk, L, lane);
            __syncwarp();
        }
        const uint32_t *walk = sm.walk;

        // draw of a site: proposal + second word stay in registers, the alias entry lands in
        // shared memory (slot `a`) through cp.async
        auto draw = [&](const PairCursor &s, uint32_t a, uint32_t &idx, uint32_t &ry) {
            idx = PAD;
            ry = 0;
            if (lane < K) {
                const uint4 r = philox4x32_10(p.seed_lo, p.seed_hi, wid_lo, wid_hi,
                                              (s.i << 16) | s.j, (TAG_NEG << 24) | lane);
                idx = __umulhi(r.x, p.n);
                ry = r.y;
                if (p.use_alias) cp_async8(sm.alias(a) + lane, p.alias + idx);
            }
        };
        auto resolve = [&](const PairCursor &s, uint32_t a, uint32_t idx, uint32_t ry,
                           uint32_t &neg) -> uint32_t {
            neg = idx;
            if (p.use_alias && lane < K) {
                const uint2 e = sm.alias(a)[lane];
                neg = ry < e.x ? idx : e.y;
            }
            const uint32_t same = __match_any_sync(FULL, neg);
            const bool valid = lane < K && neg != s.c && neg != s.o &&
                               (same & ((1u << lane) - 1u)) == 0u;
            return (__ballot_sync(FULL, valid) << 1) | 1u;
        };
        auto issue = [&](uint32_t stage, uint32_t ids, uint32_t vmask, uint32_t centre_or_pad) {
            if (vmask == full_mask) issue_rows<KP1, true>(p, sm, v, stage, lane, ids, vmask, centre_or_pad);
            else issue_rows<KP1, false>(p, sm, v, stage, lane, ids, vmask, centre_or_pad);
        };

        PairCursor scan;
        scan.i = 0xFFFFFFFFu; scan.j = 0; scan.c = PAD; scan.o = PAD; scan.hi = 0;
        bool ok_cur = next_pair<true>(p, wid_lo, wid_hi, walk, L, W, scan);
        if (!ok_cur) continue;
        PairCursor cur = scan;
        uint32_t stage = 0, slot_a = 0;

        // prologue: pair 0 synchronously, draw of pair 1 in flight
        uint32_t idx_n = PAD, ry_n = 0, neg_cur, vmask_cur, ids_cur;
        draw(cur, slot_a, idx_n, ry_n);
        cp_async_commit();
        cp_async_wait_all();
        vmask_cur = resolve(cur, slot_a, idx_n, ry_n, neg_cur);
        ids_cur = slot_ids(lane, cur.o, neg_cur, vmask_cur);
        issue(stage, ids_cur, vmask_cur, cur.c);
        bool ok_nxt = next_pair<true>(p, wid_lo, wid_hi, walk, L, W, scan);
        PairCursor nxt = scan;
        slot_a ^= 1u;
        if (ok_nxt) draw(nxt, slot_a, idx_n, ry_n);
        cp_async_commit();

        float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
        uint32_t loaded = 0xFFFFFFFFu;
        float lr = p.lr;
        while (ok_cur) {
            cp_async_wait_all();  // rows of `cur` (this stage) and alias entries of `nxt` are here
            // Memory ordering between lanes: the copies above were waited for by the lane that
            // issued them, and the ids / alias slots of the other stage were last read in the
            // previous iteration.  The warp is converged here anyway (ballot / match follow); the
            // barrier makes the ordering a guarantee of the memory model instead of a property of
            // the hardware.
            __syncwarp();
            // ---- pair p+1: resolve ids, copy its rows unless pair p is about to update one ----
            uint32_t neg_nxt = PAD, vmask_nxt = 0, ids_nxt = 0xFFFFFF00u | lane;
            bool deferred = false;
            if (ok_nxt) {
                vmask_nxt = resolve(nxt, slot_a, idx_n, ry_n, neg_nxt);
                ids_nxt = slot_ids(lane, nxt.o, neg_nxt, vmask_nxt);
                uint32_t moved = __shfl_sync(FULL, ids_nxt, lane & 15u);
                if (moved >= 0xFFFFFF00u) moved |= 16u;  // keep the two sentinel families apart
                const uint32_t both = lane < 16u ? ids_cur : moved;
                const uint32_t same = __match_any_sync(FULL, both);
                deferred = __ballot_sync(FULL, lane < 16u && (same >> 16) != 0u) != 0u ||
                           (nxt.i != cur.i && nxt.c == cur.c);
                if (!deferred) issue(stage ^ 1u, ids_nxt, vmask_nxt, nxt.i != cur.i ? nxt.c : PAD);
            }
            // ---- pair p+2: start its draw ----
            const bool ok_far = ok_nxt && next_pair<true>(p, wid_lo, wid_hi, walk, L, W, scan);
            const PairCursor far = scan;
            uint32_t idx_f = PAD, ry_f = 0;
            if (ok_far) draw(far, slot_a ^ 1u, idx_f, ry_f);
            cp_async_commit();

            // ---- pair p: train out of shared memory ----
            if (loaded != cur.i) {
                h = v.active ? lds128(sm.rows(stage) + 4u * lane + (K + 1u) * sm.pitch)
                             : make_float4(0.f, 0.f, 0.f, 0.f);
                lr = centre_lr(p, cur.c);
                loaded = cur.i;
            }
            const float4 acc = vmask_cur == full_mask
                ? train_site<KP1, true>(p, sm, v, stage, lane, vmask_cur, lr, h, loss_acc)
                : train_site<KP1, false>(p, sm, v, stage, lane, vmask_cur, lr, h, loss_acc);
            add4(h, acc);
            n_targets += __popc(vmask_cur);
            ++n_pairs;
            if ((!ok_nxt || nxt.i != cur.i) && v.active)
                *reinterpret_cast<float4 *>(const_cast<char *>(v.row0(cur.c))) = h;

            if (deferred) {  // its rows overlap the rows just stored: copy them now
                issue(stage ^ 1u, ids_nxt, vmask_nxt, nxt.i != cur.i ? nxt.c : PAD);
                cp_async_commit();
            }
            cur = nxt; neg_cur = neg_nxt; vmask_cur = vmask_nxt; ids_cur = ids_nxt; ok_cur = ok_nxt;
            nxt = far; idx_n = idx_f; ry_n = ry_f; ok_nxt = ok_far;
            stage ^= 1u;
            slot_a ^= 1u;
        }
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

// ---- K5: CBOW.  A draw site is a centre: its K+1 target rows (T1) ride the same asynchronous
// pipeline.  The <= 2W context rows (T0) of a centre are the window of the walk, and the window
// moves one position per centre: each row is needed by up to 2W consecutive centres.  So the
// warp keeps the window in a shared-memory RING indexed by walk position (2W + 2 slots: the
// 2W + 1 positions of the current window plus the one entering it): a row is copied from HBM
// once, one centre before it enters (cp.async, same commit group as the next centre's
// targets), read from shared memory for the mean, updated in place in shared memory, and its
// change is pushed to HBM as a 128-bit `red.global.add` per lane -- no read-modify-write round
// trip, and concurrent walks that share a hub row ADD their updates instead of overwriting
// each other's.  A token that occurs at two window positions owns two ring slots; they start
// equal (the second copy is issued only after the first one's pending update, like a deferred
// target copy) and receive the same sequence of additions, so they stay equal.  In the
// single-warp launch HBM and ring agree at every step, `old + acc` by the L2 atomic unit is the
// same IEEE addition the oracle performs, and the tables reproduce oracle/sgns.c bit for bit.
__device__ __forceinline__ void red_add4(float *gmem, const float4 &v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(gmem), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

__host__ __device__ __forceinline__ uint32_t cbow_ring_slots(uint32_t window) { return 2u * window + 2u; }

// FULL: the row fills all 32 lanes (embedding_size in 125..128): the per-lane "do I hold a chunk"
// predicate is then a compile-time constant
template <int KP1, bool FULL = false>
__global__ void __launch_bounds__(128, 3) cbow_pipe_kernel(const TrainParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t K = KP1 ? (uint32_t)(KP1 - 1) : p.negatives;
    const uint32_t L = p.walk_length, W = p.window;
    const uint32_t full_mask = (2u << K) - 1u;
    const uint32_t R = cbow_ring_slots(W);
    PipeSmem sm;
    float *ring;  // [R][pitch]: T0 rows of the walk positions around the centre, slot = position % R
    {
        unsigned char *base = smem_raw + warp * (pipe_warp_bytes(K, p.chunks, L) + R * p.chunks * 16u);
        sm.pitch = p.chunks * 4u;
        sm.stage_floats = (K + 2u) * sm.pitch;
        sm.rows_base = reinterpret_cast<float *>(base);
        sm.alias_base = reinterpret_cast<uint2 *>(sm.rows_base + 2u * sm.stage_floats);
        sm.ids_base = reinterpret_cast<uint32_t *>(sm.alias_base + 64);
        sm.walk = sm.ids_base + 2 * PIPE_SLOTS;
        ring = reinterpret_cast<float *>(base + pipe_warp_bytes(K, p.chunks, L));
    }
    LaneView v;
    v.t0 = reinterpret_cast<const char *>(p.t0) + 16u * lane;
    v.t1 = reinterpret_cast<const char *>(p.t1) + 16u * lane;
    v.row_bytes = p.row_stride * 4u;
    v.active = FULL ? true : lane < p.chunks;
    v.smem_chunk = FULL ? 4u * lane : 4u * (lane < p.chunks ? lane : p.chunks - 1u);
    const uint32_t lower = (1u << lane) - 1u;
    float loss_acc = 0.0f;
    unsigned long long n_pairs = 0, n_targets = 0;

    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(&p.counters->work_counter, 1ull);
        w = __shfl_sync(FULL, w, 0);
        if (w >= p.n_walks) break;
        const uint64_t wid = p.first_walk + w * p.walk_id_stride;
        const uint32_t wid_lo = (uint32_t)wid, wid_hi = (uint32_t)(wid >> 32);
        {
            const uint32_t *src = p.walks + w * (uint64_t)L;
            __syncwarp();
            for (uint32_t t = lane; t < L; t += 32u) sm.walk[t] = __ldg(src + t);
            stage_skip_mask(p, wid_lo, wid_hi, sm.walk, L, lane);
            __syncwarp();
        }
        const uint32_t *walk = sm.walk;

        auto draw = [&](uint32_t i, uint32_t a, uint32_t &idx, uint32_t &ry) {
            idx = PAD;
            ry = 0;
            if (lane < K) {
                const uint4 r = philox4x32_10(p.seed_lo, p.seed_hi, wid_lo, wid_hi,
                                              (i << 16) | 0xFFFFu, (TAG_NEG << 24) | lane);
                idx = __umulhi(r.x, p.n);
                ry = r.y;
                if (p.use_alias) cp_async8(sm.alias(a) + lane, p.alias + idx);
            }
        };
        auto resolve = [&](uint32_t c, uint32_t a, uint32_t idx, uint32_t ry, uint32_t &neg) -> uint32_t {
            neg = idx;
            if (p.use_alias && lane < K) {
                const uint2 e = sm.alias(a)[lane];
                neg = ry < e.x ? idx : e.y;
            }
            const uint32_t same = __match_any_sync(FULL, neg);
            const bool valid = lane < K && neg != c && (same & lower) == 0u;
            return (__ballot_sync(FULL, valid) << 1) | 1u;
        };
        auto issue = [&](uint32_t stage, uint32_t ids, uint32_t vmask) {
            if (vmask == full_mask) issue_rows<KP1, true>(p, sm, v, stage, lane, ids, vmask, PAD);
            else issue_rows<KP1, false>(p, sm, v, stage, lane, ids, vmask, PAD);
        };
        // Ring slot of a walk position = position mod R, kept without a division: `slot_lo` is the
        // slot of the first window position `lo_at`, and every position the loop touches lies less
        // than R behind or ahead of it.
        uint32_t lo_at = 0, slot_lo = 0;
        auto slot_of = [&](uint32_t pos) -> uint32_t {
            const uint32_t s = slot_lo + (pos - lo_at);
            return s >= R ? s - R : s;
        };
        // copy the T0 row of walk position `pos` into its ring slot (nothing to copy for PAD)
        auto fetch = [&](uint32_t pos) {
            const uint32_t t = walk[pos];
            if (t != PAD && v.active) cp_async16(ring + slot_of(pos) * sm.pitch + 4u * lane, v.row0(t));
        };

        uint32_t c_cur = PAD, c_nxt = PAD, c_far = PAD;
        uint32_t i_cur = next_centre<true>(p, wid_lo, wid_hi, walk, L, W, 0, c_cur);
        if (i_cur >= L) continue;
        uint32_t stage = 0, slot_a = 0;
        uint32_t idx_n = PAD, ry_n = 0, neg_cur, vmask_cur, ids_cur;
        draw(i_cur, slot_a, idx_n, ry_n);
        cp_async_commit();
        cp_async_wait_all();
        vmask_cur = resolve(c_cur, slot_a, idx_n, ry_n, neg_cur);
        ids_cur = slot_ids(lane, c_cur, neg_cur, vmask_cur);
        issue(stage, ids_cur, vmask_cur);
        // positions < resident are in the ring (or are PAD); the first window is copied here
        uint32_t resident = i_cur > W ? i_cur - W : 0u;
        lo_at = resident;
        slot_lo = resident % R;
        for (const uint32_t end = min(L, i_cur + W + 1u); resident < end; ++resident) fetch(resident);
        uint32_t i_nxt = next_centre<true>(p, wid_lo, wid_hi, walk, L, W, i_cur + 1, c_nxt);
        slot_a ^= 1u;
        if (i_nxt < L) draw(i_nxt, slot_a, idx_n, ry_n);
        cp_async_commit();

        while (i_cur < L) {
            cp_async_wait_all();
            __syncwarp();  // inter-lane memory ordering, see skipgram_pipe_kernel
            const uint32_t i = i_cur, c = c_cur;
            const uint32_t lo = i > W ? i - W : 0u;
            const uint32_t hi = i + W < L - 1 ? i + W : L - 1;
            {  // the window moved: usually by one position, by more after skipped centres
                const uint32_t moved = lo - lo_at;
                slot_lo = moved < R ? slot_lo + moved : (slot_lo + moved) % R;
                if (slot_lo >= R) slot_lo -= R;
                lo_at = lo;
            }
            if (resident <= hi) {  // the centre jumped (skipped centres): complete the window now
                if (resident < lo) resident = lo;
                for (; resident <= hi; ++resident) fetch(resident);
                cp_async_commit();
                cp_async_wait_all();
                __syncwarp();
            }
            // ---- the window of centre p: lane l looks at window slot l (2W + 1 <= 32) ----
            const uint32_t j = lo + lane;
            const uint32_t tok = j <= hi ? walk[j] : PAD;
            const bool ctx = j <= hi && j != i && tok != PAD && tok != c;
            const uint32_t cmask = __ballot_sync(FULL, ctx);
            const uint32_t m = __popc(cmask);
            // float offset of window slot `lane` inside the ring: the loops below fetch it by shuffle
            const uint32_t my_ring = slot_of(lo + lane) * sm.pitch;

            // ---- centre p+1: resolve ids, copy its target rows and the row entering the window ----
            uint32_t neg_nxt = PAD, vmask_nxt = 0, ids_nxt = 0xFFFFFF00u | lane;
            bool deferred = false, deferred_ring = false;
            if (i_nxt < L) {
                vmask_nxt = resolve(c_nxt, slot_a, idx_n, ry_n, neg_nxt);
                ids_nxt = slot_ids(lane, c_nxt, neg_nxt, vmask_nxt);
                uint32_t moved = __shfl_sync(FULL, ids_nxt, lane & 15u);
                if (moved >= 0xFFFFFF00u) moved |= 16u;
                const uint32_t both = lane < 16u ? ids_cur : moved;
                const uint32_t same = __match_any_sync(FULL, both);
                deferred = __ballot_sync(FULL, lane < 16u && (same >> 16) != 0u) != 0u;
                if (!deferred) issue(stage ^ 1u, ids_nxt, vmask_nxt);
                // one position ahead of the window: its slot is the spare one (2W + 2 slots)
                if (resident == hi + 1u && resident < L && resident <= i_nxt + W) {
                    const uint32_t entering = walk[resident];
                    // a row this centre is about to update would be copied stale: copy it afterwards
                    deferred_ring = __ballot_sync(FULL, ctx && tok == entering) != 0u;
                    if (!deferred_ring) fetch(resident);
                    ++resident;
                }
            }
            // ---- centre p+2: start its draw ----
            const uint32_t i_far = i_nxt < L ? next_centre<true>(p, wid_lo, wid_hi, walk, L, W, i_nxt + 1, c_far) : L;
            uint32_t idx_f = PAD, ry_f = 0;
            if (i_far < L) draw(i_far, slot_a ^ 1u, idx_f, ry_f);
            cp_async_commit();

            // ---- centre p: hidden vector = mean of the context rows, in window order ----
            const float lr = centre_lr(p, c);
            float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
            {
                bool first = true;
                for (uint32_t rem = cmask; rem; rem &= rem - 1u) {
                    const uint32_t q = __ffs(rem) - 1u;
                    const float4 r = lds128(ring + __shfl_sync(FULL, my_ring, q) + v.smem_chunk);
                    if (first) h = r; else add4(h, r);
                    first = false;
                }
                if (!v.active) h = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            const float fm = (float)m;
            h.x = __fdiv_rn(h.x, fm);
            h.y = __fdiv_rn(h.y, fm);
            h.z = __fdiv_rn(h.z, fm);
            h.w = __fdiv_rn(h.w, fm);

            const float4 acc = vmask_cur == full_mask
                ? train_site<KP1, true>(p, sm, v, stage, lane, vmask_cur, lr, h, loss_acc)
                : train_site<KP1, false>(p, sm, v, stage, lane, vmask_cur, lr, h, loss_acc);
            n_targets += __popc(vmask_cur);
            n_pairs += m;

            // ---- acc goes to every context position: in place in the ring, as an atomic add to
            //      HBM.  A token at k window positions receives k sequential additions, like the
            //      per-position oracle: every one of its slots adds acc k times, its first
            //      position issues the k atomics. ----
            {
                const uint32_t key = ctx ? tok : (0xFFFFFF00u | lane);
                const uint32_t same = __match_any_sync(FULL, key);
                const uint32_t leaders = __ballot_sync(FULL, ctx && (same & lower) == 0u);
                if (leaders == cmask) {  // every context token occurs once: the common case
                    for (uint32_t rem = cmask; rem; rem &= rem - 1u) {
                        const uint32_t q = __ffs(rem) - 1u;
                        const uint32_t t_id = __shfl_sync(FULL, tok, q);
                        const uint32_t at = __shfl_sync(FULL, my_ring, q);
                        if (v.active) {
                            float *slot = ring + at + 4u * lane;
                            float4 r = lds128(slot);
                            add4(r, acc);
                            *reinterpret_cast<float4 *>(slot) = r;
                            red_add4(reinterpret_cast<float *>(const_cast<char *>(v.row0(t_id))), acc);
                        }
                    }
                } else {
                    const uint32_t mult = __popc(same);
                    for (uint32_t rem = cmask; rem; rem &= rem - 1u) {
                        const uint32_t q = __ffs(rem) - 1u;
                        const uint32_t k = __shfl_sync(FULL, mult, q);
                        const uint32_t t_id = __shfl_sync(FULL, tok, q);
                        const uint32_t at = __shfl_sync(FULL, my_ring, q);
                        if (v.active) {
                            float *slot = ring + at + 4u * lane;
                            float4 r = lds128(slot);
                            for (uint32_t t = 0; t < k; ++t) add4(r, acc);
                            *reinterpret_cast<float4 *>(slot) = r;
                            if ((leaders >> q) & 1u)
                                for (uint32_t t = 0; t < k; ++t)
                                    red_add4(reinterpret_cast<float *>(const_cast<char *>(v.row0(t_id))), acc);
                        }
                    }
                }
            }

            if (deferred || deferred_ring) {
                if (deferred) issue(stage ^ 1u, ids_nxt, vmask_nxt);
                if (deferred_ring) fetch(resident - 1u);
                cp_async_commit();
            }
            i_cur = i_nxt; c_cur = c_nxt; neg_cur = neg_nxt; vmask_cur = vmask_nxt; ids_cur = ids_nxt;
            i_nxt = i_far; c_nxt = c_far; idx_n = idx_f; ry_n = ry_f;
            stage ^= 1u;
            slot_a ^= 1u;
        }
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

// ---- K4b (opt-in, `shared_negatives`): SkipGram with one set of negatives per CENTRE.  The m
// pairs of a centre all score against the same h = T0[c]; when they also share their K negatives
// the m x K block of negative scores collapses to K (each negative stands for m pairs, its
// gradient carries the factor m), and a centre moves m + K + 1 rows instead of m (K + 1) + 1.
// The positives are the T1 rows of the window, and the window slides: they live in the ring of
// the CBOW kernel (a row is copied from HBM once, scored and updated in shared memory by up to
// 2W centres, every update written through as one 128-bit red.global.add per lane); the K
// negatives and the centre's T0 row ride the two-stage pipeline.  Rows that the centre being
// trained is about to write (its negatives, its context rows, its own T0 row) are never copied
// early: such copies are issued after its stores, as in the kernels above.  Semantics and
// floating point: oracle/sgns.c, train_centre_shared; the single-warp launch reproduces it bit
// for bit.  Needs 2W + 1 <= 16 and K <= 15 (two id sets are compared in one MATCH).
// a stage of the shared-negative kernel holds K + 1 rows, one fewer than a stage of the per-pair
// kernels: with D = 100, K = 10, W = 4 four CTAs of four warps then fit an SM (54.6 KB each)
__host__ __device__ __forceinline__ uint32_t shared_warp_bytes(uint32_t negatives, uint32_t chunks,
                                                               uint32_t walk_length) {
    return pipe_warp_bytes(negatives, chunks, walk_length) - 2u * chunks * 16u;
}

template <int KT, int MINB = 3>
__global__ void __launch_bounds__(128, MINB) skipgram_shared_kernel(const TrainParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t K = KT ? (uint32_t)KT : p.negatives;
    const uint32_t L = p.walk_length, W = p.window;
    const uint32_t full_mask = (1u << K) - 1u;  // K ones
    const uint32_t R = cbow_ring_slots(W);
    PipeSmem sm;
    float *ring;  // [R][pitch]: T1 rows of the walk positions around the centre
    {
        unsigned char *base = smem_raw + warp * (shared_warp_bytes(K, p.chunks, L) + R * p.chunks * 16u);
        sm.pitch = p.chunks * 4u;
        sm.stage_floats = (K + 1u) * sm.pitch;  // K negatives and the centre's T0 row
        sm.rows_base = reinterpret_cast<float *>(base);
        sm.alias_base = reinterpret_cast<uint2 *>(sm.rows_base + 2u * sm.stage_floats);
        sm.ids_base = reinterpret_cast<uint32_t *>(sm.alias_base + 64);
        sm.walk = sm.ids_base + 2 * PIPE_SLOTS;
        ring = reinterpret_cast<float *>(base + shared_warp_bytes(K, p.chunks, L));
    }
    LaneView v;
    v.t0 = reinterpret_cast<const char *>(p.t0) + 16u * lane;
    v.t1 = reinterpret_cast<const char *>(p.t1) + 16u * lane;
    v.row_bytes = p.row_stride * 4u;
    v.active = lane < p.chunks;
    v.smem_chunk = 4u * (lane < p.chunks ? lane : p.chunks - 1u);
    const uint32_t lower = (1u << lane) - 1u;
    const uint32_t sentinel = 0xFFFFFF00u | lane;
    float loss_acc = 0.0f;
    unsigned long long n_pairs = 0, n_targets = 0;

    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(&p.counters->work_counter, 1ull);
        w = __shfl_sync(FULL, w, 0);
        if (w >= p.n_walks) break;
        const uint64_t wid = p.first_walk + w * p.walk_id_stride;
        const uint32_t wid_lo = (uint32_t)wid, wid_hi = (uint32_t)(wid >> 32);
        {
            const uint32_t *src = p.walks + w * (uint64_t)L;
            __syncwarp();
            for (uint32_t t = lane; t < L; t += 32u) sm.walk[t] = __ldg(src + t);
            stage_skip_mask(p, wid_lo, wid_hi, sm.walk, L, lane);
            __syncwarp();
        }
        const uint32_t *walk = sm.walk;

        auto draw = [&](uint32_t i, uint32_t a, uint32_t &idx, uint32_t &ry) {
            idx = PAD;
            ry = 0;
            if (lane < K) {
                const uint4 r = philox4x32_10(p.seed_lo, p.seed_hi, wid_lo, wid_hi,
                                              (i << 16) | 0xFFFFu, (TAG_NEG << 24) | lane);
                idx = __umulhi(r.x, p.n);
                ry = r.y;
                if (p.use_alias) cp_async8(sm.alias(a) + lane, p.alias + idx);
            }
        };
        // ids of the negatives of centre i (token c), lane k = draw k: a draw that hits the centre,
        // an earlier draw or a context token of the window is off (sentinel).  Lanes 0..15 hold
        // the window, lanes 16..16+K-1 the draws: one MATCH answers both questions.
        auto resolve = [&](uint32_t i, uint32_t c, uint32_t a, uint32_t idx, uint32_t ry, uint32_t &vmask) -> uint32_t {
            uint32_t neg = idx;
            if (p.use_alias && lane < K) {
                const uint2 e = sm.alias(a)[lane];
                neg = ry < e.x ? idx : e.y;
            }
            const uint32_t lo = i > W ? i - W : 0u;
            const uint32_t hi = i + W < L - 1 ? i + W : L - 1;
            const uint32_t moved = __shfl_sync(FULL, neg, lane & 15u);
            uint32_t key = sentinel;
            if (lane < 16u) {
                const uint32_t j = lo + lane;
                if (j <= hi && j != i) {
                    const uint32_t t = walk[j];
                    if (t != PAD && t != c) key = t;
                }
            } else if (lane - 16u < K) {
                key = moved;
            }
            const uint32_t same = __match_any_sync(FULL, key);
            const bool valid = lane >= 16u && lane - 16u < K && moved != c && (same & 0xFFFFu) == 0u &&
                               ((same >> 16) & ((1u << (lane - 16u)) - 1u)) == 0u;
            vmask = __ballot_sync(FULL, valid) >> 16;
            return ((vmask >> lane) & 1u) ? neg : sentinel;  // vmask has no bit at or above K
        };
        auto issue = [&](uint32_t stage, uint32_t ids, uint32_t vmask, uint32_t centre) {
            if (vmask == full_mask) issue_rows<KT, true, true>(p, sm, v, stage, lane, ids, vmask, centre);
            else issue_rows<KT, false, true>(p, sm, v, stage, lane, ids, vmask, centre);
        };
        uint32_t lo_at = 0, slot_lo = 0;  // ring slot of a walk position = position mod R, see cbow_pipe_kernel
        auto slot_of = [&](uint32_t pos) -> uint32_t {
            const uint32_t s = slot_lo + (pos - lo_at);
            return s >= R ? s - R : s;
        };
        auto fetch = [&](uint32_t pos) {
            const uint32_t t = walk[pos];
            if (t != PAD && v.active) cp_async16(ring + slot_of(pos) * sm.pitch + 4u * lane, v.row1(t));
        };

        uint32_t c_cur = PAD, c_nxt = PAD, c_far = PAD;
        uint32_t i_cur = next_centre<true>(p, wid_lo, wid_hi, walk, L, W, 0, c_cur);
        if (i_cur >= L) continue;
        uint32_t stage = 0, slot_a = 0;
        uint32_t idx_n = PAD, ry_n = 0, vmask_cur, ids_cur;
        draw(i_cur, slot_a, idx_n, ry_n);
        cp_async_commit();
        cp_async_wait_all();
        ids_cur = resolve(i_cur, c_cur, slot_a, idx_n, ry_n, vmask_cur);
        issue(stage, ids_cur, vmask_cur, c_cur);
        uint32_t resident = i_cur > W ? i_cur - W : 0u;  // positions < resident are in the ring (or are PAD)
        lo_at = resident;
        slot_lo = resident % R;
        for (const uint32_t end = min(L, i_cur + W + 1u); resident < end; ++resident) fetch(resident);
        uint32_t i_nxt = next_centre<true>(p, wid_lo, wid_hi, walk, L, W, i_cur + 1, c_nxt);
        slot_a ^= 1u;
        if (i_nxt < L) draw(i_nxt, slot_a, idx_n, ry_n);
        cp_async_commit();

        while (i_cur < L) {
            cp_async_wait_all();
            __syncwarp();  // inter-lane memory ordering, see skipgram_pipe_kernel
            const uint32_t i = i_cur, c = c_cur;
            const uint32_t lo = i > W ? i - W : 0u;
            const uint32_t hi = i + W < L - 1 ? i + W : L - 1;
            {
                const uint32_t moved = lo - lo_at;
                slot_lo = moved < R ? slot_lo + moved : (slot_lo + moved) % R;
                if (slot_lo >= R) slot_lo -= R;
                lo_at = lo;
            }
            if (resident <= hi) {  // the centre jumped (skipped centres): complete the window now
                if (resident < lo) resident = lo;
                for (; resident <= hi; ++resident) fetch(resident);
                cp_async_commit();
                cp_async_wait_all();
                __syncwarp();
            }
            // ---- the window of centre p: lane l looks at window slot l (2W + 1 <= 16) ----
            const uint32_t j = lo + lane;
            const uint32_t tok = j <= hi ? walk[j] : PAD;
            const bool ctx = j <= hi && j != i && tok != PAD && tok != c;
            const uint32_t cmask = __ballot_sync(FULL, ctx);
            const uint32_t m = __popc(cmask);
            const uint32_t my_ring = slot_of(lo + lane) * sm.pitch;
            const uint32_t ctx_key = ctx ? tok : sentinel;

            // ---- centre p+1: its negatives, its T0 row and the T1 row entering the window ----
            uint32_t vmask_nxt = 0, ids_nxt = sentinel;
            bool deferred = false, deferred_ring = false;
            if (i_nxt < L) {
                ids_nxt = resolve(i_nxt, c_nxt, slot_a, idx_n, ry_n, vmask_nxt);
                uint32_t moved = __shfl_sync(FULL, ids_nxt, lane & 15u);
                if (moved >= 0xFFFFFF00u) moved |= 16u;  // keep the two sentinel families apart
                // a negative of p+1 that p is about to write: as one of its negatives, as a context row
                const uint32_t hit_negs = __match_any_sync(FULL, lane < 16u ? ids_cur : moved);
                const uint32_t hit_ctx = __match_any_sync(FULL, lane < 16u ? ctx_key : moved);
                deferred = __ballot_sync(FULL, lane < 16u && ((hit_negs | hit_ctx) >> 16) != 0u) != 0u ||
                           c_nxt == c;  // ... or the same centre token again (skipped centres between)
                if (!deferred) issue(stage ^ 1u, ids_nxt, vmask_nxt, c_nxt);
                if (resident == hi + 1u && resident < L && resident <= i_nxt + W) {
                    const uint32_t entering = walk[resident];
                    deferred_ring = __ballot_sync(FULL, ctx_key == entering || ids_cur == entering) != 0u;
                    if (!deferred_ring) fetch(resident);
                    ++resident;
                }
            }
            // ---- centre p+2: start its draw ----
            const uint32_t i_far = i_nxt < L ? next_centre<true>(p, wid_lo, wid_hi, walk, L, W, i_nxt + 1, c_far) : L;
            uint32_t idx_f = PAD, ry_f = 0;
            if (i_far < L) draw(i_far, slot_a ^ 1u, idx_f, ry_f);
            cp_async_commit();

            // ---- centre p: every target is scored against h = T0[c] before anything is updated ----
            const float lr = centre_lr(p, c);
            float4 h = v.active ? lds128(sm.rows(stage) + 4u * lane + K * sm.pitch) : make_float4(0.f, 0.f, 0.f, 0.f);
            float g_mine = 0.0f;
            uint32_t applied;  // bit s: the context at window slot s is applied (a context, not clipped)
            {
                float part[16];
#pragma unroll
                for (int s = 0; s < 16; ++s) {
                    float d = 0.0f;
                    if ((cmask >> s) & 1u) {
                        const float4 r = lds128(ring + __shfl_sync(FULL, my_ring, s) + v.smem_chunk);
                        d = __fmaf_rn(h.x, r.x, d);
                        d = __fmaf_rn(h.y, r.y, d);
                        d = __fmaf_rn(h.z, r.z, d);
                        d = __fmaf_rn(h.w, r.w, d);
                    }
                    part[s] = d;
                }
                float f = reduce16(part, lane);  // lane l: score of window slot (l >> 1) & 15
                if (p.scale_dot) f = __fmul_rn(f, p.inv_scale);
                const bool my_on = (cmask >> ((lane >> 1) & 15u)) & 1u;
                bool apply = false;
                if (my_on && !(fabsf(f) > p.clip)) {
                    const float e = exp_det(-f);
                    const float sigmoid = __fdiv_rn(1.0f, __fadd_rn(1.0f, e));
                    g_mine = __fmul_rn(__fsub_rn(1.0f, sigmoid), lr);
                    if ((lane & 1u) == 0) loss_acc += __logf(1.0f + e);
                    apply = true;
                }
                // the decision for slot s sits on lanes 2s, 2s + 1: gather it to lane s
                applied = __ballot_sync(FULL, __shfl_sync(FULL, (int)apply, (2u * lane) & 31u) != 0) & 0xFFFFu & cmask;
            }
            // the K negatives: each stands for the m pairs of this centre
            const float fm = (float)m;
            const float4 acc_n = vmask_cur == full_mask
                ? train_site<KT, true, true>(p, sm, v, stage, lane, vmask_cur, lr, h, loss_acc, fm)
                : train_site<KT, false, true>(p, sm, v, stage, lane, vmask_cur, lr, h, loss_acc, fm);
            // the contexts: T1[o] += g h, in the ring and (written through) in HBM; a token at k
            // window positions receives k additions in each of its slots, its first position
            // issues the k atomics
            float4 acc_p = make_float4(0.f, 0.f, 0.f, 0.f);
            {
                const uint32_t same = __match_any_sync(FULL, ctx_key);
                const uint32_t leaders = __ballot_sync(FULL, ctx && (same & lower) == 0u);
                const uint32_t mult = __popc(same);
                // one context row: acc_p += g * row (as it was), row += k times fl(g h) here and in HBM
                auto push = [&](uint32_t q, uint32_t k, bool leader) {
                    const float g = __shfl_sync(FULL, g_mine, 2u * q);
                    const uint32_t at = __shfl_sync(FULL, my_ring, q);
                    const uint32_t t_id = __shfl_sync(FULL, tok, q);
                    if (v.active) {
                        float *slot = ring + at + 4u * lane;
                        float4 r = lds128(slot);
                        acc_p.x = __fmaf_rn(g, r.x, acc_p.x);
                        acc_p.y = __fmaf_rn(g, r.y, acc_p.y);
                        acc_p.z = __fmaf_rn(g, r.z, acc_p.z);
                        acc_p.w = __fmaf_rn(g, r.w, acc_p.w);
                        const float4 delta = make_float4(__fmul_rn(g, h.x), __fmul_rn(g, h.y), __fmul_rn(g, h.z),
                                                         __fmul_rn(g, h.w));
                        float *row = reinterpret_cast<float *>(const_cast<char *>(v.row1(t_id)));
                        if (k == 1u) {
                            add4(r, delta);
                            red_add4(row, delta);
                        } else {
                            for (uint32_t t = 0; t < k; ++t) add4(r, delta);
                            if (leader)
                                for (uint32_t t = 0; t < k; ++t) red_add4(row, delta);
                        }
                        *reinterpret_cast<float4 *>(slot) = r;
                    }
                };
                if (leaders == cmask) {  // every context token occurs once: the common case
                    for (uint32_t rem = applied; rem; rem &= rem - 1u) push(__ffs(rem) - 1u, 1u, true);
                } else {
                    for (uint32_t rem = applied; rem; rem &= rem - 1u) {
                        const uint32_t q = __ffs(rem) - 1u;
                        push(q, __shfl_sync(FULL, mult, q), (leaders >> q) & 1u);
                    }
                }
            }
            add4(acc_p, acc_n);
            add4(h, acc_p);
            if (v.active) *reinterpret_cast<float4 *>(const_cast<char *>(v.row0(c))) = h;
            n_targets += __popc(vmask_cur) + m;
            n_pairs += m;

            if (deferred || deferred_ring) {
                if (deferred) issue(stage ^ 1u, ids_nxt, vmask_nxt, c_nxt);
                if (deferred_ring) fetch(resident - 1u);
                cp_async_commit();
            }
            i_cur = i_nxt; c_cur = c_nxt; vmask_cur = vmask_nxt; ids_cur = ids_nxt;
            i_nxt = i_far; c_nxt = c_far; idx_n = idx_f; ry_n = ry_f;
            stage ^= 1u;
            slot_a ^= 1u;
        }
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

bool shared_negatives_supported(const TrainParams &p) {
    return p.chunks <= 32u && p.negatives <= 15u && 2u * p.window + 1u <= 16u && p.walk_length <= 1024u;
}

bool pipe_supported(const TrainParams &p, uint32_t model) {
    if (p.chunks > 32u || p.negatives + 1u > PIPE_SLOTS || p.walk_length > 1024u) return false;
    return model == B2E_SKIPGRAM || 2u * p.window + 1u <= 32u;
}

template <typename Kernel>
static cudaError_t launch_pipe(Kernel kernel, const TrainParams &p, bool deterministic, int sm_count,
                               uint64_t max_warps, cudaStream_t stream, size_t extra_warp_bytes = 0,
                               int max_per_sm = 0) {
    const size_t warp_bytes = pipe_warp_bytes(p.negatives, p.chunks, p.walk_length) + extra_warp_bytes;
    const int warps = deterministic ? 1 : 4;
    const size_t smem = warp_bytes * warps;
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (err != cudaSuccess) return err;
    if (deterministic) {
        kernel<<<1, 32, smem, stream>>>(p);
        return cudaGetLastError();
    }
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 128, smem);
    if (err != cudaSuccess) return err;
    if (per_sm < 1) per_sm = 1;
    if (max_per_sm && per_sm > max_per_sm) per_sm = max_per_sm;
    uint64_t grid = (uint64_t)sm_count * per_sm;  // persistent: every CTA resident, walks fetched
    const uint64_t needed = (std::min<uint64_t>(p.n_walks, max_warps) + warps - 1) / warps;
    if (grid > needed) grid = needed;
    if (grid < 1) grid = 1;
    kernel<<<(unsigned)grid, 128, smem, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_train_pipe(const TrainParams &p, uint32_t model, bool deterministic, int sm_count,
                              uint64_t max_warps, cudaStream_t stream) {
    cudaError_t err = cudaMemsetAsync(&p.counters->work_counter, 0, sizeof(unsigned long long), stream);
    if (err != cudaSuccess) return err;
    if (model == B2E_SKIPGRAM && p.shared_negatives) {
        if (!shared_negatives_supported(p)) return cudaErrorInvalidValue;  // b2e_create refuses these
        // launch_pipe sizes a warp's slab as pipe_warp_bytes + extra: one row per stage less here
        const size_t ring = (size_t)cbow_ring_slots(p.window) * p.chunks * 16u - 2u * p.chunks * 16u;
        switch (p.negatives) {
            case 10:
                // four CTAs per SM (128 registers, 54.6 KB each) rather than three: the kernel is bound
                // by the dependency chain of a warp, not by HBM -- C3 2.61 G against 2.20 G pairs/s, C5
                // 2.51 G (profiles/r02x_*)
                if (!deterministic)
                    return launch_pipe(skipgram_shared_kernel<10, 4>, p, deterministic, sm_count, max_warps, stream, ring);
                return launch_pipe(skipgram_shared_kernel<10>, p, deterministic, sm_count, max_warps, stream, ring);
            case 5: return launch_pipe(skipgram_shared_kernel<5>, p, deterministic, sm_count, max_warps, stream, ring);
            default: return launch_pipe(skipgram_shared_kernel<0>, p, deterministic, sm_count, max_warps, stream, ring);
        }
    }
    // CTAs per SM of the SkipGram kernel, measured in pairs/s at 5 / 4 / 3 / 2 with a switch since
    // removed: C2 543 / 605 / 596 / -, C3 537 / 587 / 583 / -, C5 473 / 503 / 516 / 460 M
    // (profiles/r02p_*): four while the tables are a few GB, three once random rows spread over
    // tens of GB (fewer streams keep more DRAM pages open); the switch-over is put at 32 GiB of tables.
    const bool large_tables = 2ull * p.n * p.row_stride * sizeof(float) >= (32ull << 30);
    if (model == B2E_SKIPGRAM && large_tables && p.negatives + 1u == 11u && !deterministic)
        return launch_pipe(skipgram_pipe_kernel<11, 3>, p, deterministic, sm_count, max_warps, stream, 0, 3);
    if (model == B2E_SKIPGRAM) {
        switch (p.negatives + 1u) {
            case 11: return launch_pipe(skipgram_pipe_kernel<11>, p, deterministic, sm_count, max_warps, stream);
            case 6: return launch_pipe(skipgram_pipe_kernel<6>, p, deterministic, sm_count, max_warps, stream);
            default: return launch_pipe(skipgram_pipe_kernel<0>, p, deterministic, sm_count, max_warps, stream);
        }
    }
    const size_t ring = (size_t)cbow_ring_slots(p.window) * p.chunks * 16u;
    if (p.chunks == 32u && p.negatives + 1u == 11u)
        return launch_pipe(cbow_pipe_kernel<11, true>, p, deterministic, sm_count, max_warps, stream, ring);
    switch (p.negatives + 1u) {
        case 11: return launch_pipe(cbow_pipe_kernel<11>, p, deterministic, sm_count, max_warps, stream, ring);
        case 6: return launch_pipe(cbow_pipe_kernel<6>, p, deterministic, sm_count, max_warps, stream, ring);
        default: return launch_pipe(cbow_pipe_kernel<0>, p, deterministic, sm_count, max_warps, stream, ring);
    }
}

}  // namespace b2e
