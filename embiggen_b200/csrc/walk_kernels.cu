// K2: DeepWalk / node2vec walk kernels for sm_100a.
//
// Replaces the walk half of `ensmallen.models.SkipGram/CBOW.fit_transform`
// (/root/reference/embiggen/embedders/ensmallen_embedders/node2vec.py:99; walk kwargs
// .../node2vec_skipgram.py:51-81).  One walk per thread: a walk is a chain of dependent
// random 32 B-sector gathers (offsets -> neighbour), so throughput comes from the number of
// independent chains in flight per SM, not from wide loads.  Second order uses KnightKing
// rejection sampling against a uniform neighbour proposal with an integer accept test, so the
// result is bit-identical to the CPU oracle driven by the same Philox stream.
//
// Tokens are buffered four at a time in registers and written with one 16 B store: two
// consecutive stores fill a 32 B sector while the line is still resident in L2.
#include <algorithm>

#include "common.cuh"

namespace b2e {

// sorted-row membership by lower-bound bisection; every load is counted as one probe
template <typename Count>
__device__ __forceinline__ bool row_contains(const uint32_t *__restrict__ row, uint32_t len,
                                             uint32_t key, Count &probes) {
    uint32_t lo = 0, hi = len;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        ++probes;
        if (__ldg(row + mid) < key) lo = mid + 1; else hi = mid;
    }
    if (lo >= len) return false;
    ++probes;
    return __ldg(row + lo) == key;
}

// ---- row filters: a blocked Bloom filter per neighbour list ----
//
// The adjacency check "is x a neighbour of prev" decides between the COMMON and EXPLORE classes.
// On a sparse graph the answer is almost always "no", and finding that out by bisecting a sorted
// hub row costs log2(deg) dependent sector gathers.  A filter answers most of them with ONE
// 8-byte gather: one byte of filter per directed edge, laid over the row's own edge range --
// row v owns the 32 B sectors that bytes [indptr[v], indptr[v + 1]) touch, so no second offset
// array is needed (boundary sectors are shared with the neighbouring rows, which can only set
// more bits) -- a key picks one sector by hash, one of its four words, and three bits in it.
// No false negatives: "not in the filter" is final; "maybe" falls through to the exact search.
// Rows shorter than FILTER_MIN_DEG are searched directly (one or two sectors).  The filter never
// changes a decision, so the walks stay bit-identical to the oracle, which has no filter.
constexpr uint32_t FILTER_MIN_DEG = 16;
constexpr uint32_t SHORT_ROW_MIN_DEG = 64;  // from here on fetch the proposal's row and bisect the shorter

__host__ __device__ __forceinline__ uint32_t fmix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
    return h;
}

struct FilterSlot { uint64_t word; unsigned long long mask; };

__device__ __forceinline__ FilterSlot filter_slot(int64_t off, uint32_t deg, uint32_t key) {
    const uint64_t first = (uint64_t)off >> 5, last = ((uint64_t)off + deg - 1u) >> 5;
    const uint32_t h1 = fmix32(key), h2 = fmix32(key ^ 0x9E3779B9u);
    const uint64_t sector = first + __umulhi(h1, (uint32_t)(last - first) + 1u);
    FilterSlot s;
    s.word = sector * 4u + (h2 & 3u);
    s.mask = (1ull << ((h2 >> 2) & 63u)) | (1ull << ((h2 >> 8) & 63u)) | (1ull << ((h2 >> 14) & 63u));
    return s;
}

uint64_t row_filter_words(uint64_t nnz) { return ((nnz + 31u) / 32u) * 4u + 4u; }

// lane l looks at row base + l; rows of at least `min_deg` edges are then walked by the whole warp
template <typename RowFn, typename EdgeFn>
__device__ __forceinline__ void for_each_row(const int64_t *__restrict__ indptr, uint64_t n, uint32_t min_deg,
                                             RowFn small_row, EdgeFn edge) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t base = (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32u; base < n;
         base += warps * 32u) {
        const uint64_t v = base + lane;
        int64_t off = 0;
        uint32_t deg = 0;
        if (v < n) {
            off = __ldg(indptr + v);
            deg = (uint32_t)(__ldg(indptr + v + 1) - off);
        }
        const bool big = deg >= min_deg;
        if (!big && deg) small_row(v, off, deg);
        uint32_t todo = __ballot_sync(0xffffffffu, big);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1u;
            const int64_t o = __shfl_sync(0xffffffffu, off, src);
            const uint32_t d = __shfl_sync(0xffffffffu, deg, src);
            for (uint32_t e = lane; e < d; e += 32u) edge(base + src, o, d, e);
        }
    }
}

__global__ void __launch_bounds__(256) row_filter_build_kernel(const int64_t *__restrict__ indptr,
                                                               const uint32_t *__restrict__ indices, uint64_t n,
                                                               unsigned long long *filter) {
    for_each_row(indptr, n, FILTER_MIN_DEG, [](uint64_t, int64_t, uint32_t) {},
                 [&](uint64_t, int64_t off, uint32_t deg, uint32_t e) {
                     const FilterSlot s = filter_slot(off, deg, __ldg(indices + off + e));
                     atomicOr(filter + s.word, s.mask);
                 });
}

cudaError_t launch_row_filter_build(const int64_t *indptr, const uint32_t *indices, uint64_t n,
                                    unsigned long long *filter, int sm_count, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)sm_count * 16);
    row_filter_build_kernel<<<grid, 256, 0, stream>>>(indptr, indices, n, filter);
    return cudaGetLastError();
}

// Every destination id below n and every row strictly ascending?  The walk kernels, the symmetry
// check and the SGD kernels index with these ids without looking again.
__global__ void __launch_bounds__(256) csr_check_kernel(const int64_t *__restrict__ indptr,
                                                        const uint32_t *__restrict__ indices, uint64_t n,
                                                        int *flags) {
    int bad = 0;
    for_each_row(indptr, n, 32u,
                 [&](uint64_t, int64_t off, uint32_t deg) {
                     uint32_t last = __ldg(indices + off);
                     if (last >= n) bad |= 1;
                     for (uint32_t e = 1; e < deg; ++e) {
                         const uint32_t x = __ldg(indices + off + e);
                         if (x >= n) bad |= 1;
                         if (x <= last) bad |= 2;
                         last = x;
                     }
                 },
                 [&](uint64_t, int64_t off, uint32_t deg, uint32_t e) {
                     const uint32_t x = __ldg(indices + off + e);
                     if (x >= n) bad |= 1;
                     if (e + 1u < deg && __ldg(indices + off + e + 1) <= x) bad |= 2;
                 });
    if (bad) atomicOr(flags, bad);
}

cudaError_t launch_csr_check(const int64_t *indptr, const uint32_t *indices, uint64_t n, int *d_flags,
                             int sm_count, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)sm_count * 16);
    csr_check_kernel<<<grid, 256, 0, stream>>>(indptr, indices, n, d_flags);
    return cudaGetLastError();
}

// Is x a neighbour of prev?  Filter first, then the exact search: on an undirected graph
// (x in N(prev) <=> prev in N(x)) the shorter of the two rows is bisected, and the bounds of
// x's row, fetched for that, are handed back so that an accepted x does not fetch them again.
struct RowBounds { int64_t off; uint32_t deg; bool valid; };

template <typename Count>
__device__ __forceinline__ bool adjacent(const WalkParams &p, int64_t prev_off, uint32_t prev_deg,
                                         uint32_t prev, uint32_t x, RowBounds &xrow,
                                         Count &probes, Count &rejects) {
    if (p.filter && prev_deg >= FILTER_MIN_DEG) {
        const FilterSlot s = filter_slot(prev_off, prev_deg, x);
        ++probes;
        if ((__ldg(p.filter + s.word) & s.mask) != s.mask) {
            ++rejects;
            return false;
        }
    }
    if (p.undirected && prev_deg >= SHORT_ROW_MIN_DEG) {
        xrow.off = __ldg(p.indptr + x);
        xrow.deg = (uint32_t)(__ldg(p.indptr + x + 1) - xrow.off);
        xrow.valid = true;
        ++probes;
        if (xrow.deg < prev_deg) return row_contains(p.indices + xrow.off, xrow.deg, prev, probes);
    }
    return row_contains(p.indices + prev_off, prev_deg, x, probes);
}

// index of a proposal inside a row: uniform, or proportional to the edge weights through the
// row's Vose alias table built at load time -- O(1): one 8-byte gather; the high word of r * deg
// picks the slot, its low word is the coin (oracle/walks.c: propose)
template <bool WEIGHTED>
__device__ __forceinline__ uint32_t propose(const uint2 *__restrict__ table, int64_t off, uint32_t deg,
                                            uint32_t r) {
    const unsigned long long u = (unsigned long long)r * deg;
    const uint32_t i = (uint32_t)(u >> 32);
    if (!WEIGHTED) return i;
    const uint2 e = __ldg(table + off + i);
    return (uint32_t)u < e.x ? i : e.y;
}

// FOLD (unweighted, undirected, return_weight > max(1, explore_weight)): the return edge is cut
// down to the envelope of the other classes and its excess becomes a virtual slot of the row --
// one Philox block per trial (tag 12): x decides slot vs row, y proposes, z accepts; see
// oracle/walks.c (orc_fold_thresholds) for the normative statement.
// MINB: resident CTAs per SM the register allocation is held to (4: 64 registers, no spills;
// 6: 40 registers and a few spilled words -- more chains in flight per SM).  The vectorised
// second-order unweighted walks use 6: on C3 they ran at 7.8 / 8.6 / 9.4 G steps/s at 4 / 5 / 6
// and 9.3 at 8 (profiles/r02c_*, r02d_bench_c3_occ8, measured with a switch since removed).
template <bool SECOND, bool VEC, bool WEIGHTED, bool FOLD, int MINB = 4>
__global__ void __launch_bounds__(256, MINB) walk_kernel(const WalkParams p) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // per-thread counts stay far below 2^32 (L < 2^16 steps, at most 2^20 trials each is a cap
    // never approached); they are widened when the warp adds them up
    uint32_t n_steps = 0, n_trials = 0, n_searches = 0;
    uint32_t n_probes = 0, n_rejects = 0;
    if (i < p.n_walks) {
        const uint64_t wid = p.first_walk + i * p.walk_id_stride;
        const uint32_t wid_lo = (uint32_t)wid, wid_hi = (uint32_t)(wid >> 32);
        uint32_t *out = p.out + i * (uint64_t)p.walk_length;
        const unsigned long long thr_lo = min(p.thr_common, p.thr_explore);
        const unsigned long long thr_hi = max(p.thr_common, p.thr_explore);
        const uint32_t L = p.walk_length;

        uint32_t cur = __ldg(p.sources + (wid % p.n_src));
        int64_t prev_off = 0;
        uint32_t prev = PAD, prev_deg = 0;
        RowBounds row = {0, 0, false};  // bounds of cur's row when an adjacency check already fetched them
        uint4 rnd = make_uint4(0, 0, 0, 0);
        uint4 tok = make_uint4(cur, PAD, PAD, PAD);  // four tokens leave as one 16-byte store
        bool alive = true;
        for (uint32_t t = 1; t < L; ++t) {
            uint32_t next = PAD;
            if (alive) {
                int64_t off;
                uint32_t deg;
                if (SECOND && row.valid) {
                    off = row.off;
                    deg = row.deg;
                } else {
                    off = __ldg(p.indptr + cur);
                    deg = (uint32_t)(__ldg(p.indptr + cur + 1) - off);
                }
                row.valid = false;
                if (deg == 0) {
                    alive = false;
                } else {
                    if (!SECOND || t == 1) {
                        const uint32_t s = t - 1;
                        if ((s & 3u) == 0 || (SECOND && t == 1))
                            rnd = philox4x32_10(p.seed_lo, p.seed_hi, wid_lo, wid_hi, s >> 2, TAG_WALK1 << 24);
                        const uint32_t r = (s & 3u) == 0 ? rnd.x : (s & 3u) == 1 ? rnd.y
                                         : (s & 3u) == 2 ? rnd.z : rnd.w;
                        next = __ldg(p.indices + off + propose<WEIGHTED>(p.edge_alias, off, deg, r));
                    } else {
                        const unsigned long long t_out =
                            FOLD ? (p.fold_excess << 32) / (((unsigned long long)deg << 20) + p.fold_excess) : 0ull;
                        uint32_t trial = 0;
                        for (;;) {
                            uint32_t r0;
                            unsigned long long r1;
                            ++n_trials;
                            if constexpr (FOLD) {
                                rnd = philox4x32_10(p.seed_lo, p.seed_hi, wid_lo, wid_hi, t - 1,
                                                    (TAG_FOLD << 24) | trial);
                                if (rnd.x < t_out) {  // the virtual slot: back to where we came from
                                    next = prev;
                                    row.off = prev_off;
                                    row.deg = prev_deg;
                                    row.valid = true;
                                    break;
                                }
                                r0 = rnd.y;
                                r1 = rnd.z;
                            } else {
                                if ((trial & 1u) == 0)
                                    rnd = philox4x32_10(p.seed_lo, p.seed_hi, wid_lo, wid_hi, t - 1,
                                                        (TAG_WALK2 << 24) | (trial >> 1));
                                r0 = (trial & 1u) ? rnd.z : rnd.x;
                                r1 = (trial & 1u) ? rnd.w : rnd.y;
                            }
                            next = __ldg(p.indices + off + propose<WEIGHTED>(p.edge_alias, off, deg, r0));
                            bool accept;
                            RowBounds xrow = {0, 0, false};
                            if (next == prev) {
                                accept = r1 < p.thr_return;
                                xrow.off = prev_off;
                                xrow.deg = prev_deg;
                                xrow.valid = true;
                            } else if (r1 < thr_lo) {
                                accept = true;   // every non-return class accepts
                            } else if (r1 >= thr_hi) {
                                accept = false;  // every non-return class rejects
                            } else {
                                ++n_searches;
                                const bool common = adjacent(p, prev_off, prev_deg, prev, next, xrow,
                                                             n_probes, n_rejects);
                                accept = r1 < (common ? p.thr_common : p.thr_explore);
                            }
                            if (accept) { row = xrow; break; }
                            ++trial;
                            if (trial >= MAX_TRIALS) break;
                        }
                    }
                    ++n_steps;
                    prev = cur;
                    prev_off = off;
                    prev_deg = deg;
                    cur = next;
                }
            }
            const uint32_t slot = t & 3u;  // explicit selects keep the group in registers
            if (slot == 0) tok.x = next; else if (slot == 1) tok.y = next;
            else if (slot == 2) tok.z = next; else tok.w = next;
            if (slot == 3u) {
                if (VEC) {
                    *reinterpret_cast<uint4 *>(out + t - 3u) = tok;
                } else {
                    out[t - 3u] = tok.x; out[t - 2u] = tok.y; out[t - 1u] = tok.z; out[t] = tok.w;
                }
            }
        }
        const uint32_t tail = L & 3u;  // tokens of an unfinished group (never with VEC: L % 4 == 0)
        if (tail) {
            out[L - tail] = tok.x;
            if (tail > 1) out[L - tail + 1u] = tok.y;
            if (tail > 2) out[L - tail + 2u] = tok.z;
        }
    }
    // one atomic per warp and counter
    unsigned long long steps = n_steps, trials = n_trials, searches = n_searches, probes = n_probes,
                       rejects = n_rejects;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        steps += __shfl_xor_sync(0xffffffffu, steps, off);
        trials += __shfl_xor_sync(0xffffffffu, trials, off);
        searches += __shfl_xor_sync(0xffffffffu, searches, off);
        probes += __shfl_xor_sync(0xffffffffu, probes, off);
        rejects += __shfl_xor_sync(0xffffffffu, rejects, off);
    }
    if ((threadIdx.x & 31) == 0 && p.counters) {
        atomicAdd(&p.counters->walk_steps, steps);
        if (SECOND) {
            atomicAdd(&p.counters->walk_trials, trials);
            atomicAdd(&p.counters->walk_searches, searches);
            atomicAdd(&p.counters->walk_probes, probes);
            atomicAdd(&p.counters->walk_filter_rejects, rejects);
        }
    }
}


// Typed walks (change_node_type_weight / change_edge_type_weight, .../node2vec_skipgram.py:72-77):
// every transition is a trial loop with ONE Philox block per trial (tag 7): x proposal, z
// node-type test, w edge-type test, y p/q test.  Independent words => the acceptance probability
// is the product of the three ratios.  Cheap tests first; see oracle/walks.c:walks_general.
// (normalize_by_degree needs no kernel: it is folded into the proposal table at load.)
template <bool VEC, bool WEIGHTED>
__global__ void __launch_bounds__(256) walk_general_kernel(const WalkParams p) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long n_steps = 0, n_trials = 0, n_searches = 0, n_probes = 0, n_rejects = 0;
    if (i < p.n_walks) {
        const uint64_t wid = p.first_walk + i * p.walk_id_stride;
        const uint32_t wid_lo = (uint32_t)wid, wid_hi = (uint32_t)(wid >> 32);
        uint32_t *out = p.out + i * (uint64_t)p.walk_length;
        const unsigned long long thr_lo = min(p.thr_common, p.thr_explore);
        const unsigned long long thr_hi = max(p.thr_common, p.thr_explore);
        const bool use_nt = p.node_types != nullptr && p.q_node[0] != p.q_node[1];
        const bool use_et = p.edge_types != nullptr && p.q_edge[0] != p.q_edge[1];
        uint32_t cur = __ldg(p.sources + (wid % p.n_src));
        int64_t prev_off = 0;
        uint32_t prev = PAD, prev_deg = 0, prev_etype = 0;
        bool alive = true;
        uint32_t tok[4];
        const uint32_t L = p.walk_length;
        for (uint32_t base = 0; base < L; base += 4) {
#pragma unroll
            for (uint32_t u = 0; u < 4; ++u) {
                const uint32_t t = base + u;
                if (t == 0) { tok[0] = cur; continue; }
                if (t >= L) { tok[u] = PAD; continue; }
                uint32_t next = PAD;
                if (alive) {
                    const int64_t off = __ldg(p.indptr + cur);
                    const uint32_t deg = (uint32_t)(__ldg(p.indptr + cur + 1) - off);
                    if (deg == 0) {
                        alive = false;
                    } else {
                        const uint32_t cur_type = use_nt ? __ldg(p.node_types + cur) : 0u;
                        uint32_t trial = 0;
                        int64_t e = off;
                        for (;;) {
                            const uint4 rnd = philox4x32_10(p.seed_lo, p.seed_hi, wid_lo, wid_hi, t - 1,
                                                            (TAG_WALK3 << 24) | trial);
                            e = off + propose<WEIGHTED>(p.edge_alias, off, deg, rnd.x);
                            next = __ldg(p.indices + e);
                            ++n_trials;
                            bool accept = true;
                            if (use_nt)
                                accept = rnd.z < p.q_node[__ldg(p.node_types + next) != cur_type ? 1 : 0];
                            if (accept && use_et && t > 1)
                                accept = rnd.w < p.q_edge[__ldg(p.edge_types + e) != prev_etype ? 1 : 0];
                            if (accept && t > 1) {
                                const unsigned long long lhs = rnd.y;
                                if (next == prev) {
                                    accept = lhs < p.thr_return;
                                } else if (lhs < thr_lo) {
                                    accept = true;
                                } else if (lhs >= thr_hi) {
                                    accept = false;
                                } else {
                                    ++n_searches;
                                    RowBounds xrow = {0, 0, false};
                                    const bool common = adjacent(p, prev_off, prev_deg, prev, next, xrow,
                                                                 n_probes, n_rejects);
                                    accept = lhs < (common ? p.thr_common : p.thr_explore);
                                }
                            }
                            if (accept) break;
                            ++trial;
                            if (trial >= MAX_TRIALS) break;
                        }
                        ++n_steps;
                        if (p.edge_types) prev_etype = __ldg(p.edge_types + e);
                        prev = cur;
                        prev_off = off;
                        prev_deg = deg;
                        cur = next;
                    }
                }
                tok[u] = next;
            }
            if (VEC) {
                *reinterpret_cast<uint4 *>(out + base) = make_uint4(tok[0], tok[1], tok[2], tok[3]);
            } else {
#pragma unroll
                for (uint32_t u = 0; u < 4; ++u)
                    if (base + u < L) out[base + u] = tok[u];
            }
        }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        n_steps += __shfl_xor_sync(0xffffffffu, n_steps, off);
        n_trials += __shfl_xor_sync(0xffffffffu, n_trials, off);
        n_searches += __shfl_xor_sync(0xffffffffu, n_searches, off);
        n_probes += __shfl_xor_sync(0xffffffffu, n_probes, off);
        n_rejects += __shfl_xor_sync(0xffffffffu, n_rejects, off);
    }
    if ((threadIdx.x & 31) == 0 && p.counters) {
        atomicAdd(&p.counters->walk_steps, n_steps);
        atomicAdd(&p.counters->walk_trials, n_trials);
        atomicAdd(&p.counters->walk_searches, n_searches);
        atomicAdd(&p.counters->walk_probes, n_probes);
        atomicAdd(&p.counters->walk_filter_rejects, n_rejects);
    }
}

// Walklets (.../walklets.py:7-149): scale k keeps the pairs exactly k hops apart, i.e. adjacent
// tokens of the k sub-walks made of every k-th token.  out[r][w][m] = raw[w][r + m k] (PAD past
// the end), sub-walk length ceil(L / k); the SGD kernels then run unchanged on the sub-walks.
__global__ void __launch_bounds__(256) walklet_split_kernel(const uint32_t *__restrict__ raw, uint64_t n_walks,
                                                            uint32_t L, uint32_t k, uint32_t Ls,
                                                            uint32_t *__restrict__ out) {
    const uint64_t total = n_walks * k * Ls;
    for (uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t m = (uint32_t)(idx % Ls);
        const uint64_t rest = idx / Ls;
        const uint64_t w = rest % n_walks;
        const uint32_t r = (uint32_t)(rest / n_walks);
        const uint32_t t = r + m * k;
        out[idx] = t < L ? __ldg(raw + w * L + t) : PAD;
    }
}

cudaError_t launch_walklet_split(const uint32_t *raw, uint64_t n_walks, uint32_t walk_length, uint32_t scale,
                                 uint32_t *out, cudaStream_t stream) {
    const uint32_t Ls = (walk_length + scale - 1) / scale;
    const uint64_t total = n_walks * scale * Ls;
    if (total == 0) return cudaSuccess;
    const uint64_t grid = std::min<uint64_t>((total + 255) / 256, 148ull * 16);
    walklet_split_kernel<<<(unsigned)grid, 256, 0, stream>>>(raw, n_walks, walk_length, scale, Ls, out);
    return cudaGetLastError();
}

// One thread per directed edge (u, v): is u in the row of v?  Clears *symmetric otherwise.
__global__ void __launch_bounds__(256) symmetry_kernel(const int64_t *__restrict__ indptr,
                                                       const uint32_t *__restrict__ indices, uint64_t n,
                                                       uint64_t nnz, int *symmetric) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz || *symmetric == 0) return;
    uint64_t lo = 0, hi = n;  // row of edge e: last u with indptr[u] <= e
    while (lo < hi) {
        const uint64_t mid = lo + ((hi - lo + 1) >> 1);
        if ((uint64_t)__ldg(indptr + mid) <= e) lo = mid; else hi = mid - 1;
    }
    const uint32_t u = (uint32_t)lo, v = __ldg(indices + e);
    const int64_t begin = __ldg(indptr + v);
    const uint32_t len = (uint32_t)(__ldg(indptr + v + 1) - begin);
    unsigned long long probes = 0;
    if (!row_contains(indices + begin, len, u, probes)) *symmetric = 0;
}

cudaError_t launch_symmetry_check(const int64_t *indptr, const uint32_t *indices, uint64_t n,
                                  uint64_t nnz, int *d_flag, cudaStream_t stream) {
    if (nnz == 0) return cudaSuccess;
    symmetry_kernel<<<(unsigned)((nnz + 255) / 256), 256, 0, stream>>>(indptr, indices, n, nnz, d_flag);
    return cudaGetLastError();
}

cudaError_t launch_walks(const WalkParams &p, bool second_order, cudaStream_t stream) {
    if (p.n_walks == 0) return cudaSuccess;
    const unsigned block = 256;
    const unsigned grid = (unsigned)((p.n_walks + block - 1) / block);
    const bool vec = (p.walk_length % 4u) == 0 && (reinterpret_cast<uintptr_t>(p.out) % 16u) == 0;
    const bool weighted = p.edge_alias != nullptr;
    const bool typed = (p.node_types && p.q_node[0] != p.q_node[1]) ||
                       (p.edge_types && p.q_edge[0] != p.q_edge[1]);
    if (typed) {  // typed walks: one trial loop per transition
        if (vec) { if (weighted) walk_general_kernel<true, true><<<grid, block, 0, stream>>>(p);
                   else walk_general_kernel<true, false><<<grid, block, 0, stream>>>(p); }
        else { if (weighted) walk_general_kernel<false, true><<<grid, block, 0, stream>>>(p);
               else walk_general_kernel<false, false><<<grid, block, 0, stream>>>(p); }
        return cudaGetLastError();
    }
#define B2E_LAUNCH_WALK(...) walk_kernel<__VA_ARGS__><<<grid, block, 0, stream>>>(p)
    if (second_order && !weighted && vec) {  // the headline shapes, six CTAs per SM
        if (p.fold_excess) B2E_LAUNCH_WALK(true, true, false, true, 6); else B2E_LAUNCH_WALK(true, true, false, false, 6);
    } else if (second_order && !weighted) {
        if (p.fold_excess) B2E_LAUNCH_WALK(true, false, false, true); else B2E_LAUNCH_WALK(true, false, false, false);
    } else if (second_order) {
        if (vec) B2E_LAUNCH_WALK(true, true, true, false); else B2E_LAUNCH_WALK(true, false, true, false);
    } else {
        if (vec) { if (weighted) B2E_LAUNCH_WALK(false, true, true, false); else B2E_LAUNCH_WALK(false, true, false, false); }
        else { if (weighted) B2E_LAUNCH_WALK(false, false, true, false); else B2E_LAUNCH_WALK(false, false, false, false); }
    }
#undef B2E_LAUNCH_WALK
    return cudaGetLastError();
}

}  // namespace b2e
