// Approximate batched search (sm_100a): for a query q of length m and a budget e <= kMaxMismatches, every window start p
// with p + m <= n and Hamming(T[p, p+m), q) <= e, ascending. Substitutions only.
//
// Pigeonhole seeds: L = floor(m / (e+1)); seed j is the query segment [jL, (j+1)L), j = 0..e. A window within e
// substitutions matches at least one of these e+1 disjoint segments exactly. Seed j is looked up as
//   * the k-mer at query offset jL of the element with the largest k <= L (an auxiliary k' = L element included): its
//     bucket lists every x with T[x, x+k) == q[jL, jL+k), or, when every k is larger than L,
//   * the whole segment through the prefix slab of the element with the smallest k > L (the buckets of all k-mers that
//     start with it, bounded by lower_bound_key as the sub-k plan of search_kernels.cu does) plus the k - L starts at the
//     end of the text where no k-mer starts, compared directly.
// Candidate x of seed j gives p = x - jL. Seed i lists p exactly when T[p+iL, ...) equals its seed, so p is dropped when
// an earlier seed i < j matches there: every window is verified once, by its first error-free seed, and no sort or
// dedup pass is needed. Survivors are verified with mismatches_span on the packed text (early exit above e).
// One group of G lanes per query, as the general search kernel; two passes (count -> scan -> write); candidate lists
// longer than kHeavyCandidates go to a warp-per-query launch. Hits of several seeds, or of a slab, are not ascending:
// such a query is flagged for launch_segment_sort.
//
// Hit strategies (kmer_b200_approx_hits) other than "all" start with a best pass (kApproxBest): the count-pass
// enumeration of every query with budget min(e, m - 1), each lane keeping the smallest (d << 32 | p) of its survivors;
// it writes d_min and the lowest position with that distance, and lists the queries that have one. Single-best ends
// there (one hit per listed query, launch_approx_single). All-best and strata run the count and write passes again
// over the listed queries only (kApproxListed), each with its own budget e_q = min(e, d_min + s): the e_q + 1 seeds
// enumerate exactly the windows with d <= e_q. launch_approx_distances recomputes d(p) of every written hit.
//
// Collection index (COLL, args.approx == 2): a window counts only when it lies inside one record (window_in_record on
// the boundary bitmap), checked where a verified window becomes a hit or a lane's best, so every pass and strategy sees
// in-record windows only. The check depends on p alone, so the first-error-free-seed dedup stays exact. The kernels of
// a plain index are instantiated without it.
#include <algorithm>

#include "launch.h"
#include "query_pack.cuh"

namespace kb {

constexpr int kApproxThreads = 256;

// PASS: kPassCount, kPassCountAccount (count + gathered sectors) or kPassWrite. HEAVY: the warp-per-query launch over
// the heavy list. MODE: kApproxAll (budget a.max_mismatches, every query), kApproxListed (budget h.budget[q], the
// queries of a.hits; the count pass does not list them again) or kApproxBest (count passes only: the best pass).
template <int PASS_, int G, bool HEAVY, int MODE = kApproxAll, bool COLL = false>
__device__ __forceinline__ void approx_query(const SearchArgs &a, const uint64_t q, uint64_t *smem_q,
                                             const ApproxHitArgs &h = ApproxHitArgs{}) {
    constexpr bool kAccount = PASS_ == kPassCountAccount;
    constexpr int PASS = kAccount ? (int)kPassCount : PASS_;
    constexpr bool kBest = MODE == kApproxBest;
    const int lane = threadIdx.x & 31;
    const int gl = threadIdx.x & (G - 1);
    const int group = threadIdx.x / G;
    const uint32_t gshift = (uint32_t)(lane - gl);
    const uint32_t gfull = G == 32 ? 0xFFFFFFFFu : ((1u << G) - 1);
    const uint32_t gmask = gfull << gshift;
    const uint32_t lt_mask = (1u << gl) - 1;
#define GBALLOT(pred) (G == 1 ? ((pred) ? 1u : 0u) : ((__ballot_sync(gmask, (pred)) >> gshift) & gfull))
#define GSHFL(v, src) (G == 1 ? (v) : __shfl_sync(gmask, (v), (src), G))
// the count pass enlists a query with a long candidate list for the warp launch (marked in unsorted[q] bit 1); the
// write pass follows that mark. Both passes see the same lookups, hence the same decision.
#define HAND_OFF_IF_HEAVY(len)                                                                          \
    if (PASS == kPassCount && !HEAVY && G < 32 && a.heavy != nullptr && (len) > (uint64_t)kHeavyCandidates) { \
        if (gl == 0) {                                                                                  \
            a.heavy[1 + atomicAdd(a.heavy, 1u)] = (uint32_t)q;                                          \
            a.counts[q] = 0;                                                                            \
            a.status[q] = KMER_B200_QUERY_OK;                                                           \
            a.unsorted[q] = 2;                                                                          \
        }                                                                                               \
        return;                                                                                         \
    }

    uint64_t out_base = 0;
    if (PASS == kPassWrite) {
        out_base = a.counts[q];
        if (a.counts[q + 1] == out_base) return;
        if (!HEAVY && G < 32 && (a.unsorted[q] & 2)) return;
    }
    const DeviceIndex &ix = *a.index;
    const PackedText T = ix.text;
    const uint64_t off0 = a.q_offsets[q];
    const uint64_t m64 = a.q_offsets[q + 1] - off0;
    uint32_t e = MODE == kApproxListed ? (uint32_t)h.budget[q] : a.max_mismatches;
    uint32_t status = KMER_B200_QUERY_OK;
    if (m64 == 0) status = KMER_B200_QUERY_UNDEFINED;
    else if (m64 > a.max_len) status = KMER_B200_QUERY_TOO_LONG_FOR_SHARD;  // longer than the caller's max_query_len
    if (status != KMER_B200_QUERY_OK) {
        if (PASS == kPassCount && gl == 0) {
            a.counts[q] = 0;
            a.status[q] = (uint8_t)status;
            a.unsorted[q] = 0;
            if (kBest) h.best_dist[q] = 0xFF;
        }
        return;
    }
    const uint32_t m = (uint32_t)m64;
    if (kBest && e >= m) e = m - 1;  // d_min of a query of m <= e symbols: below m if a window is found, else m
    uint64_t best = ~0ull;           // kApproxBest: this lane's smallest (d << 32 | p)
    uint64_t *qw = smem_q + (size_t)group * a.q_words;
    pack_query_group<G>(a.q_ranks, off0, m, a.q_offsets[a.n_queries], T, (uint32_t)gl, gmask, a.error_flag, qw);

    uint32_t n_gather = 0;
    uint64_t n_hits = 0;
    bool unsorted = false;
    if (m <= e || (uint64_t)m > T.n) {
        // every window is within e substitutions of a query of at most e symbols (or no window fits); on a collection
        // the in-record ones: counted from the table, written by scanning every window start
        const uint64_t n_win = (uint64_t)m > T.n ? 0 : (COLL ? ix.n_win[m] : T.n - m + 1);
        HAND_OFF_IF_HEAVY(n_win)
        n_hits = n_win;
        if (PASS == kPassWrite && !COLL)
            for (uint64_t p = gl; p < n_win; p += G) a.positions[out_base + p] = (uint32_t)p;
        if (PASS == kPassWrite && COLL) {
            uint64_t k = 0;
            for (uint64_t p0 = 0; p0 + m <= T.n && k < n_win; p0 += G) {
                const uint64_t p = p0 + gl;
                const bool ok = p + m <= T.n && window_in_record(ix.boundary, p, m);
                const uint32_t b = GBALLOT(ok);
                if (ok) a.positions[out_base + k + __popc(b & lt_mask)] = (uint32_t)p;
                k += __popc(b);
            }
        }
    } else {
        const uint32_t L = m / (e + 1);
        // the seed element: the largest k <= L, else the smallest k (> L), enumerated as prefix slabs
        uint32_t es = ix.elem_by_k_desc[ix.n_elems - 1];
        bool slab = true;
        for (uint32_t i = 0; i < ix.n_elems; ++i) {
            const uint32_t c = ix.elem_by_k_desc[i];
            if (ix.elem[c].k <= L) {
                es = c;
                slab = false;
                break;
            }
        }
        if (L < 64 && ix.aux_for_len[L] != 0xFF && (slab || ix.elem[es].k < L)) {
            es = ix.aux_for_len[L];
            slab = false;
        }
        const Element &E = ix.elem[es];
        const uint32_t s_len = slab ? L : E.k;      // symbols of a seed that its candidates match exactly
        const uint32_t n_tail = slab ? E.k - L : 0;  // per slab seed: starts behind the last k-mer, compared directly

        // ---- the e+1 lookups: independent, issued together (lane j % G takes seed j)
        Range sr[kMaxMismatches + 1];
        uint64_t total = 0;
#pragma unroll
        for (uint32_t j = 0; j <= kMaxMismatches; ++j) {
            sr[j] = Range{0, 0};
            if (j <= e && (G == 1 || j % G == (uint32_t)gl)) {
                if (slab) {
                    const uint64_t width = ix.pow_sigma[E.k - L];
                    const uint64_t key = key_at(qw, (uint64_t)j * L, L, T.bits, T.sigma) * width;
                    const uint64_t lo = lower_bound_key(E, key);
                    sr[j] = Range{lo, lower_bound_key(E, key + width) - lo};
                    if (kAccount) n_gather += 2;
                } else {
                    sr[j] = bucket_of(E, key_at(qw, (uint64_t)j * L, E.k, T.bits, T.sigma));
                    if (kAccount) n_gather += 1 + (E.shift ? 1 : 0);
                }
                total += sr[j].cnt + n_tail;
            }
        }
        for (int o = G >> 1; o > 0; o >>= 1) total += __shfl_xor_sync(gmask, total, o, G);
        HAND_OFF_IF_HEAVY(total)

        // ---- candidates, seed by seed
        uint32_t seeds_with_hits = 0;
        for (uint32_t j = 0; j <= e; ++j) {
            const uint64_t lo = GSHFL(sr[j].lo, (int)(j % G));
            const uint64_t cnt = GSHFL(sr[j].cnt, (int)(j % G));
            const uint64_t n_cand = cnt + n_tail;
            const uint32_t so = j * L;  // the seed's query offset
            uint64_t hits_j = 0;
            for (uint64_t c0 = 0; c0 < n_cand; c0 += G) {
                const uint64_t c = c0 + gl;
                uint64_t p = 0;
                bool ok = false;
                if (c < n_cand) {
                    uint64_t x;
                    if (c < cnt) {
                        x = gather32(pos_ptr(E, lo + c));  // a slab spans buckets, so it may span parts
                        ok = true;
                        if (kAccount && (((lo + c) & 7) == 0 || c == 0)) ++n_gather;
                    } else {
                        x = T.n - E.k + 1 + (c - cnt);
                        ok = match_span(T, qw, x, so, L);
                        if (kAccount) ++n_gather;
                    }
                    ok = ok && x >= so && x - so + m <= T.n;
                    p = x - so;
                    // an earlier seed that matches exactly here has listed p already
                    for (uint32_t i = 0; ok && i < j; ++i) {
                        ok = !match_span(T, qw, p + (uint64_t)i * L, i * L, s_len);
                        if (kAccount) ++n_gather;
                    }
                    if (ok) {
                        if (kBest) {
                            // the limit follows this lane's best distance: equal distances are still counted exactly
                            const uint32_t lim = best == ~0ull ? e : (uint32_t)(best >> 32);
                            const uint32_t d = mismatches_span(T, qw, p, 0, m, lim);
                            bool in = d <= lim;
                            if (COLL && in) {
                                in = window_in_record(ix.boundary, p, m);
                                if (kAccount) ++n_gather;
                            }
                            if (in) best = min(best, ((uint64_t)d << 32) | p);
                            ok = false;
                        } else {
                            ok = mismatches_span(T, qw, p, 0, m, e) <= e;
                            if (COLL && ok) {
                                ok = window_in_record(ix.boundary, p, m);
                                if (kAccount) ++n_gather;
                            }
                        }
                        if (kAccount) n_gather += 1 + (m * T.bits >> 8);
                    }
                }
                const uint32_t b = GBALLOT(ok);
                if (PASS == kPassWrite && ok) a.positions[out_base + n_hits + __popc(b & lt_mask)] = (uint32_t)p;
                n_hits += __popc(b);
                hits_j += __popc(b);
            }
            seeds_with_hits += hits_j != 0 ? 1u : 0u;
        }
        unsorted = seeds_with_hits > 1 || slab;  // a bucket of one seed is ascending; a slab is ordered by hash
    }
    if (kAccount) {
        for (int o = G >> 1; o > 0; o >>= 1) n_gather += __shfl_xor_sync(gmask, n_gather, o, G);
        if (gl == 0) atomicAdd(a.gather_count, (unsigned long long)n_gather);
    }
    if (kBest) {
        for (int o = G >> 1; o > 0; o >>= 1) best = min(best, (uint64_t)__shfl_xor_sync(gmask, best, o, G));
        if (best == ~0ull && m <= a.max_mismatches && (uint64_t)m <= T.n) {
            // every window: d = m, lowest at 0 (on a collection: at the first in-record window, if any)
            if (!COLL) best = (uint64_t)m << 32;
            else if (ix.n_win[m] != 0) best = ((uint64_t)m << 32) | ix.first_win[m];
        }
        if (gl == 0) {
            const bool found = best != ~0ull;
            const uint32_t d = (uint32_t)(best >> 32);
            a.counts[q] = found ? 1 : 0;
            a.status[q] = KMER_B200_QUERY_OK;
            a.unsorted[q] = HEAVY ? 2 : 0;
            h.best_dist[q] = found ? (uint8_t)d : (uint8_t)0xFF;
            h.best_pos[q] = (uint32_t)best;
            if (h.budget && found) h.budget[q] = (uint8_t)min(a.max_mismatches, d + h.strata);
            if (found) a.hits[1 + atomicAdd(a.hits, 1u)] = (uint32_t)q;
        }
        return;
    }
    if (PASS == kPassCount && gl == 0) {
        a.counts[q] = n_hits;
        a.status[q] = KMER_B200_QUERY_OK;
        const bool flag = unsorted && n_hits > 1;
        a.unsorted[q] = (flag ? 1 : 0) | (HEAVY ? 2 : 0);
        if (flag) atomicAdd(a.error_flag + 1, 1u);  // number of segments the sort pass has to visit
        if (MODE == kApproxAll && a.hits != nullptr && n_hits > 0) {
            // the write pass only visits the queries listed here
            const uint32_t act = __activemask();
            const int leader = __ffs(act) - 1;
            uint32_t slot = 0;
            if (lane == leader) slot = atomicAdd(a.hits, (uint32_t)__popc(act));
            slot = __shfl_sync(act, slot, leader) + __popc(act & ((1u << lane) - 1));
            a.hits[1 + slot] = (uint32_t)q;
        }
    }
#undef HAND_OFF_IF_HEAVY
#undef GBALLOT
#undef GSHFL
}

// count pass: one group per query; write pass (and every pass of kApproxListed): the queries the count pass listed as
// having hits
template <int PASS, int G, int MODE, bool COLL = false>
__device__ __forceinline__ void approx_grid(const SearchArgs &a, const ApproxHitArgs &h, uint64_t *smem_q) {
    constexpr int kGroups = kApproxThreads / G;
    if ((PASS == kPassWrite || MODE == kApproxListed) && a.hits != nullptr) {
        const uint32_t n_listed = a.hits[0];
        for (uint64_t i = (uint64_t)blockIdx.x * kGroups + threadIdx.x / G; i < n_listed; i += (uint64_t)gridDim.x * kGroups) {
            approx_query<PASS, G, false, MODE, COLL>(a, (uint64_t)a.hits[1 + i], smem_q, h);
            __syncwarp();
        }
    } else {
        const uint64_t q = (uint64_t)blockIdx.x * kGroups + threadIdx.x / G;
        if (q < a.n_queries) approx_query<PASS, G, false, MODE, COLL>(a, q, smem_q, h);
    }
}

template <int PASS, int G>
__global__ void __launch_bounds__(kApproxThreads) search_approx_kernel(const SearchArgs a) {
    extern __shared__ uint64_t smem_q[];
    approx_grid<PASS, G, kApproxAll>(a, ApproxHitArgs{}, smem_q);
}

template <int PASS, int G, int MODE>
__global__ void __launch_bounds__(kApproxThreads) search_approx_hits_kernel(const SearchArgs a, const ApproxHitArgs h) {
    extern __shared__ uint64_t smem_q[];
    approx_grid<PASS, G, MODE>(a, h, smem_q);
}

// second launch of a pass: one warp per query of the heavy list (a.heavy[0] = length, a.heavy[1..] = query ids)
template <int PASS, int MODE, bool COLL = false>
__device__ __forceinline__ void approx_heavy(const SearchArgs &a, const ApproxHitArgs &h, uint64_t *smem_q) {
    constexpr int kGroups = kApproxThreads / 32;
    const uint32_t n_heavy = a.heavy[0];
    for (uint32_t i = blockIdx.x * kGroups + threadIdx.x / 32; i < n_heavy; i += gridDim.x * kGroups) {
        approx_query<PASS, 32, true, MODE, COLL>(a, (uint64_t)a.heavy[1 + i], smem_q, h);
        __syncwarp();
    }
}

template <int PASS>
__global__ void __launch_bounds__(kApproxThreads) search_approx_heavy_kernel(const SearchArgs a) {
    extern __shared__ uint64_t smem_q[];
    approx_heavy<PASS, kApproxAll>(a, ApproxHitArgs{}, smem_q);
}

template <int PASS, int MODE>
__global__ void __launch_bounds__(kApproxThreads) search_approx_heavy_hits_kernel(const SearchArgs a, const ApproxHitArgs h) {
    extern __shared__ uint64_t smem_q[];
    approx_heavy<PASS, MODE>(a, h, smem_q);
}

// every pass and mode of a collection index (approx == 2)
template <int PASS, int G, int MODE>
__global__ void __launch_bounds__(kApproxThreads) search_approx_coll_kernel(const SearchArgs a, const ApproxHitArgs h) {
    extern __shared__ uint64_t smem_q[];
    approx_grid<PASS, G, MODE, true>(a, h, smem_q);
}

template <int PASS, int MODE>
__global__ void __launch_bounds__(kApproxThreads) search_approx_heavy_coll_kernel(const SearchArgs a, const ApproxHitArgs h) {
    extern __shared__ uint64_t smem_q[];
    approx_heavy<PASS, MODE, true>(a, h, smem_q);
}

template <int PASS, int G, int MODE>
static void launch_approx_pg(const SearchArgs &args, const ApproxHitArgs &h, cudaStream_t stream) {
    constexpr int kGroups = kApproxThreads / G;
    const size_t smem = (size_t)kGroups * args.q_words * sizeof(uint64_t);
    uint64_t blocks = (args.n_queries + kGroups - 1) / kGroups;
    if ((PASS == kPassWrite || MODE == kApproxListed) && args.hits != nullptr)
        blocks = std::min<uint64_t>(blocks, (uint64_t)device_sm_count() * 16);
    const bool coll = args.approx == 2;
    if (coll) {
        cudaFuncSetAttribute(search_approx_coll_kernel<PASS, G, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        search_approx_coll_kernel<PASS, G, MODE><<<(unsigned)blocks, kApproxThreads, smem, stream>>>(args, h);
    } else if (MODE == kApproxAll) {
        cudaFuncSetAttribute(search_approx_kernel<PASS, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        search_approx_kernel<PASS, G><<<(unsigned)blocks, kApproxThreads, smem, stream>>>(args);
    } else {
        cudaFuncSetAttribute(search_approx_hits_kernel<PASS, G, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        search_approx_hits_kernel<PASS, G, MODE><<<(unsigned)blocks, kApproxThreads, smem, stream>>>(args, h);
    }
    if (G < 32 && args.heavy != nullptr) {
        // queries with long candidate lists, if any (the list length lives on the device: fixed grid, no host sync)
        SearchArgs ha = args;
        ha.q_words = search_q_words(32, args.bits, args.max_len);
        const size_t hsmem = (size_t)(kApproxThreads / 32) * ha.q_words * sizeof(uint64_t);
        if (coll) {
            cudaFuncSetAttribute(search_approx_heavy_coll_kernel<PASS, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem);
            search_approx_heavy_coll_kernel<PASS, MODE><<<device_sm_count() * 2, kApproxThreads, hsmem, stream>>>(ha, h);
        } else if (MODE == kApproxAll) {
            cudaFuncSetAttribute(search_approx_heavy_kernel<PASS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem);
            search_approx_heavy_kernel<PASS><<<device_sm_count() * 2, kApproxThreads, hsmem, stream>>>(ha);
        } else {
            cudaFuncSetAttribute(search_approx_heavy_hits_kernel<PASS, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem);
            search_approx_heavy_hits_kernel<PASS, MODE><<<device_sm_count() * 2, kApproxThreads, hsmem, stream>>>(ha, h);
        }
    }
}

template <int G, int MODE>
static void launch_approx_g(const SearchArgs &args, const ApproxHitArgs &h, SearchPass pass, cudaStream_t stream) {
    if (pass == kPassCount) launch_approx_pg<kPassCount, G, MODE>(args, h, stream);
    if (pass == kPassCountAccount) launch_approx_pg<kPassCountAccount, G, MODE>(args, h, stream);
    if constexpr (MODE != kApproxBest)
        if (pass == kPassWrite) launch_approx_pg<kPassWrite, G, MODE>(args, h, stream);
}

template <int MODE>
static void launch_approx_m(const SearchArgs &args, const ApproxHitArgs &h, SearchPass pass, cudaStream_t stream) {
    if (args.n_queries == 0) return;
    if (args.group == 1) launch_approx_g<1, MODE>(args, h, pass, stream);
    else if (args.group == 2) launch_approx_g<2, MODE>(args, h, pass, stream);
    else if (args.group == 4) launch_approx_g<4, MODE>(args, h, pass, stream);
    else if (args.group == 8) launch_approx_g<8, MODE>(args, h, pass, stream);
    else launch_approx_g<32, MODE>(args, h, pass, stream);
}

void launch_search_approx(const SearchArgs &args, SearchPass pass, cudaStream_t stream) {
    launch_approx_m<kApproxAll>(args, ApproxHitArgs{}, pass, stream);
}

void launch_search_approx_hits(const SearchArgs &args, const ApproxHitArgs &h, ApproxMode mode, SearchPass pass,
                               cudaStream_t stream) {
    if (mode == kApproxBest) launch_approx_m<kApproxBest>(args, h, pass, stream);
    else if (mode == kApproxListed) launch_approx_m<kApproxListed>(args, h, pass, stream);
    else launch_approx_m<kApproxAll>(args, h, pass, stream);
}

// single best: the one hit of each listed query at its offset (the scan of counts = found)
__global__ void __launch_bounds__(256) approx_single_kernel(const uint32_t *__restrict__ hits, const uint64_t *__restrict__ offsets,
                                                            const uint32_t *__restrict__ best_pos, const uint8_t *__restrict__ best_dist,
                                                            uint32_t *__restrict__ positions, uint8_t *__restrict__ distances) {
    const uint32_t n = hits[0];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t q = hits[1 + i];
        const uint64_t o = offsets[q];
        positions[o] = best_pos[q];
        if (distances) distances[o] = best_dist[q];
    }
}

void launch_approx_single(const SearchArgs &args, const ApproxHitArgs &h, uint8_t *d_distances, cudaStream_t stream) {
    if (args.n_queries == 0) return;
    const uint64_t blocks = std::min<uint64_t>((args.n_queries + 255) / 256, (uint64_t)device_sm_count() * 8);
    approx_single_kernel<<<(unsigned)blocks, 256, 0, stream>>>(args.hits, args.counts, h.best_pos, h.best_dist, args.positions,
                                                               d_distances);
}

// d(p) of every written hit of the listed queries, in position order: one group per query packs it again and counts the
// mismatches of each of its windows (limit e_q: every written hit is within it, so the count is exact)
template <int G, bool ACCOUNT>
__global__ void __launch_bounds__(kApproxThreads) approx_distances_kernel(const SearchArgs a, const ApproxHitArgs h,
                                                                          uint8_t *__restrict__ distances) {
    constexpr int kGroups = kApproxThreads / G;
    extern __shared__ uint64_t smem_q[];
    const int lane = threadIdx.x & 31;
    const int gl = threadIdx.x & (G - 1);
    const uint32_t gfull = G == 32 ? 0xFFFFFFFFu : ((1u << G) - 1);
    const uint32_t gmask = gfull << (uint32_t)(lane - gl);
    uint64_t *qw = smem_q + (size_t)(threadIdx.x / G) * a.q_words;
    const PackedText T = a.index->text;
    const uint32_t n_listed = a.hits[0];
    for (uint64_t i = (uint64_t)blockIdx.x * kGroups + threadIdx.x / G; i < n_listed; i += (uint64_t)gridDim.x * kGroups) {
        const uint64_t q = a.hits[1 + i];
        const uint64_t o0 = a.counts[q], o1 = a.counts[q + 1];
        if (o0 == o1) continue;
        const uint64_t off0 = a.q_offsets[q];
        const uint32_t m = (uint32_t)(a.q_offsets[q + 1] - off0);
        const uint32_t e = h.budget ? (uint32_t)h.budget[q] : a.max_mismatches;
        pack_query_group<G>(a.q_ranks, off0, m, a.q_offsets[a.n_queries], T, (uint32_t)gl, gmask, a.error_flag, qw);
        uint32_t n_gather = 0;
        for (uint64_t j = o0 + gl; j < o1; j += G) {
            distances[j] = (uint8_t)mismatches_span(T, qw, a.positions[j], 0, m, e);
            if (ACCOUNT) n_gather += 1 + (m * T.bits >> 8);
        }
        if (ACCOUNT) {
            for (int o = G >> 1; o > 0; o >>= 1) n_gather += __shfl_xor_sync(gmask, n_gather, o, G);
            if (gl == 0) atomicAdd(a.gather_count, (unsigned long long)n_gather);
        }
        __syncwarp();
    }
}

template <int G>
static void launch_distances_g(const SearchArgs &args, const ApproxHitArgs &h, uint8_t *d_distances, cudaStream_t stream) {
    constexpr int kGroups = kApproxThreads / G;
    const size_t smem = (size_t)kGroups * args.q_words * sizeof(uint64_t);
    const uint64_t blocks = std::min<uint64_t>((args.n_queries + kGroups - 1) / kGroups, (uint64_t)device_sm_count() * 16);
    if (args.gather_count) {
        cudaFuncSetAttribute(approx_distances_kernel<G, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        approx_distances_kernel<G, true><<<(unsigned)blocks, kApproxThreads, smem, stream>>>(args, h, d_distances);
    } else {
        cudaFuncSetAttribute(approx_distances_kernel<G, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        approx_distances_kernel<G, false><<<(unsigned)blocks, kApproxThreads, smem, stream>>>(args, h, d_distances);
    }
}

void launch_approx_distances(const SearchArgs &args, const ApproxHitArgs &h, uint8_t *d_distances, cudaStream_t stream) {
    if (args.n_queries == 0) return;
    if (args.group == 1) launch_distances_g<1>(args, h, d_distances, stream);
    else if (args.group == 2) launch_distances_g<2>(args, h, d_distances, stream);
    else if (args.group == 4) launch_distances_g<4>(args, h, d_distances, stream);
    else if (args.group == 8) launch_distances_g<8>(args, h, d_distances, stream);
    else launch_distances_g<32>(args, h, d_distances, stream);
}

// ---- collection index: the record boundary bitmap (built once per attach or load) and locating hits

__global__ void __launch_bounds__(256) record_boundaries_kernel(const uint64_t *__restrict__ starts, uint64_t n_records, uint64_t n,
                                                                unsigned long long *__restrict__ bits) {
    for (uint64_t r = 1 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_records; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t s = starts[r];
        if (s > 0 && s < n) atomicOr(bits + (s >> 6), 1ull << (s & 63));
    }
}

void launch_record_boundaries(const uint64_t *d_starts, uint64_t n_records, uint64_t n, uint64_t *d_bits, cudaStream_t stream) {
    if (n_records < 2) return;
    const uint64_t blocks = std::min<uint64_t>((n_records + 255) / 256, (uint64_t)device_sm_count() * 8);
    record_boundaries_kernel<<<(unsigned)blocks, 256, 0, stream>>>(d_starts, n_records, n, (unsigned long long *)d_bits);
}

// record = the last r with starts[r] <= p (empty records share their start with the next one), offset = p - starts[r];
// a position at or past the end of the text gives (UINT32_MAX, 0)
__global__ void __launch_bounds__(256) locate_kernel(const uint64_t *__restrict__ starts, uint64_t n_records,
                                                     const uint32_t *__restrict__ positions, uint64_t n_pos,
                                                     uint32_t *__restrict__ record_out, uint32_t *__restrict__ offset_out) {
    const uint64_t n = __ldg(starts + n_records);
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pos; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t p = positions[i];
        if (p >= n) {
            record_out[i] = 0xFFFFFFFFu;
            offset_out[i] = 0;
            continue;
        }
        uint64_t lo = 0, hi = n_records;  // starts[lo] <= p < starts[hi]
        while (hi - lo > 1) {
            const uint64_t mid = (lo + hi) >> 1;
            if (__ldg(starts + mid) <= p) lo = mid;
            else hi = mid;
        }
        record_out[i] = (uint32_t)lo;
        offset_out[i] = (uint32_t)(p - __ldg(starts + lo));
    }
}

void launch_locate(const uint64_t *d_starts, uint64_t n_records, const uint32_t *d_positions, uint64_t n_pos, uint32_t *d_record,
                   uint32_t *d_offset, cudaStream_t stream) {
    if (n_pos == 0) return;
    const uint64_t blocks = std::min<uint64_t>((n_pos + 255) / 256, (uint64_t)device_sm_count() * 16);
    locate_kernel<<<(unsigned)blocks, 256, 0, stream>>>(d_starts, n_records, d_positions, n_pos, d_record, d_offset);
}

}  // namespace kb
