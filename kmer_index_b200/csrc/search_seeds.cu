// Batched k-mer seeding (sm_100a): for each query q of length m and each offset j in [0, m - k], every text position p
// with T[p, p+k) == q[j, j+k), in (j, p) order, plus the occurrence count of every k-mer of the batch.
//
// One warp per query walks its k-mers in tiles of kSeedTileSymbols symbols: the tile is packed into shared memory with
// pack_query_group (which also checks the ranks), and lane t of a round hashes the k-mer at tile offset t with key_at and
// looks it up with bucket_of. A bucket lists the k-mer's occurrences in ascending position order, so a query's hits
// need no sort: the buckets of its k-mers, taken in j order, are the (j, p) order.
//
// Count pass (seed_count_kernel): kmer_counts[i] = the occurrence count of k-mer i (saturated at max_occ + 1 when a cap
// is set), bucket_lo[i] = its first CSR entry (kept so that the write pass neither packs, hashes nor looks up again),
// counts[q] = the sum of the uncapped counts, which launch_offsets_scan turns into offsets. On a collection index a
// k-mer's count is its in-record occurrences: its bucket is walked with window_in_record, stopping at max_occ + 1 when a
// cap is set.
//
// Write pass (seed_write_kernel): the warp rescans the counts of its query's k-mers 32 at a time (a shuffle scan per
// round gives each k-mer its output offset), then copies each bucket into positions with j into seed_offsets. Buckets of
// at most kSeedLaneCopy hits are copied by their own lane, longer ones by the whole warp, and buckets of more than
// kHeavyCandidates hits go to a list that seed_heavy_kernel copies with a warp each and several loads in flight. On a
// collection index the out-of-record windows are compacted out with ballots, in order, until the k-mer's in-record
// count has been written.
#include <algorithm>

#include "launch.h"
#include "query_pack.cuh"

namespace kb {

namespace {

constexpr int kSeedThreads = 256;
constexpr int kSeedWarps = kSeedThreads / 32;
constexpr uint32_t kSeedTileSymbols = 256;                // one round of pack_query_group<32>: 8 symbols per lane
constexpr uint32_t kSeedTileWords = kSeedTileSymbols / 8 + 2;  // 8-bit symbols + the two zero words
constexpr uint32_t kSeedLaneCopy = 4;                     // buckets up to this size are copied by their own lane
constexpr uint32_t kFull = 0xFFFFFFFFu;

// inclusive warp scan
__device__ __forceinline__ uint64_t warp_scan(uint64_t v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t u = __shfl_up_sync(kFull, v, o);
        if (lane >= o) v += u;
    }
    return v;
}

__device__ __forceinline__ uint64_t warp_sum(uint64_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// in-record occurrences among the bucket entries [lo, lo + cnt) of element E, counted up to `stop` (one lane)
template <bool ACCOUNT>
__device__ __forceinline__ uint64_t in_record_lane(const SeedArgs &a, const Element &E, uint64_t lo, uint64_t cnt, uint64_t stop,
                                                   uint32_t *n_gather) {
    const uint64_t *boundary = a.index->boundary;
    uint64_t c = 0;
    for (uint64_t t = 0; t < cnt && c < stop; ++t) {
        c += window_in_record(boundary, gather32(pos_ptr(E, lo + t)), a.k) ? 1 : 0;
        if (ACCOUNT) *n_gather += 1 + ((lo + t) % 8 == 0 || t == 0 ? 1 : 0);
    }
    return c;
}

// the same with the whole warp, 32 entries per round (every lane passes the same lo, cnt, stop)
template <bool ACCOUNT>
__device__ __forceinline__ uint64_t in_record_warp(const SeedArgs &a, const Element &E, uint64_t lo, uint64_t cnt, uint64_t stop,
                                                   int lane, uint32_t *n_gather) {
    const uint64_t *boundary = a.index->boundary;
    uint64_t c = 0;
    for (uint64_t t0 = 0; t0 < cnt && c < stop; t0 += 32) {
        const uint64_t t = t0 + lane;
        bool ok = false;
        if (t < cnt) {
            ok = window_in_record(boundary, gather32(pos_ptr(E, lo + t)), a.k);
            if (ACCOUNT) *n_gather += 1 + ((lo + t) % 8 == 0 || t == 0 ? 1 : 0);
        }
        c += __popc(__ballot_sync(kFull, ok));
    }
    return min(c, stop);
}

template <bool COLL, bool ACCOUNT>
__global__ void __launch_bounds__(kSeedThreads) seed_count_kernel(const SeedArgs a) {
    __shared__ uint64_t smem_q[kSeedWarps][kSeedTileWords];
    const int lane = threadIdx.x & 31;
    const uint64_t q = (uint64_t)blockIdx.x * kSeedWarps + threadIdx.x / 32;
    if (q >= a.n_queries) return;
    const DeviceIndex &ix = *a.index;
    const PackedText T = ix.text;
    const Element &E = ix.elem[a.elem];
    uint64_t *qw = smem_q[threadIdx.x / 32];
    const uint64_t off0 = a.q_offsets[q];
    const uint64_t m = a.q_offsets[q + 1] - off0;
    const uint64_t i0 = a.kmer_base[q];
    const uint32_t k = a.k;
    const uint64_t stop = a.max_occ ? (uint64_t)a.max_occ + 1 : ~0ull;  // a count above max_occ is reported as max_occ + 1
    const uint32_t step = kSeedTileSymbols - (k - 1);                    // k-mers per full tile
    uint64_t total = 0, heavy = 0;
    uint32_t n_gather = 0;
    for (uint64_t j0 = 0; j0 < m; j0 += step) {
        const uint32_t ts = (uint32_t)min((uint64_t)kSeedTileSymbols, m - j0);
        pack_query_group<32>(a.q_ranks, off0 + j0, ts, a.q_offsets[a.n_queries], T, (uint32_t)lane, kFull, a.error_flag, qw);
        const uint32_t nk = ts >= k ? ts - k + 1 : 0;
        for (uint32_t t0 = 0; t0 < nk; t0 += 32) {
            const uint32_t t = t0 + lane;
            Range r{0, 0};
            if (t < nk) {
                r = bucket_of(E, key_at(qw, (uint64_t)t, k, T.bits, T.sigma));
                if (ACCOUNT) n_gather += 1 + (E.shift ? 1 : 0);
            }
            uint64_t c = r.cnt;
            if (COLL) {
                // short buckets are walked by their own lane, long ones by the whole warp, one after the other
                const bool big = r.cnt > 32;
                if (!big) c = in_record_lane<ACCOUNT>(a, E, r.lo, r.cnt, stop, &n_gather);
                uint32_t todo = __ballot_sync(kFull, big);
                while (todo) {
                    const int src = __ffs(todo) - 1;
                    todo &= todo - 1;
                    const uint64_t lo = __shfl_sync(kFull, r.lo, src), cnt = __shfl_sync(kFull, r.cnt, src);
                    const uint64_t cw = in_record_warp<ACCOUNT>(a, E, lo, cnt, stop, lane, &n_gather);
                    if (lane == src) c = cw;
                }
            }
            if (t < nk) {
                const uint64_t i = i0 + j0 + t;
                const bool capped = c > (a.max_occ ? (uint64_t)a.max_occ : ~0ull);
                a.kmer_counts[i] = (uint32_t)min(c, stop);
                if (a.bucket_lo) a.bucket_lo[i] = (uint32_t)r.lo;
                if (!capped) {
                    total += c;
                    heavy += c > kHeavyCandidates ? 1 : 0;
                }
            }
        }
        __syncwarp();  // the tile is read by every lane before the next one is packed over it
        if (j0 + ts >= m) break;
    }
    total = warp_sum(total);
    heavy = warp_sum(heavy);
    if (ACCOUNT) n_gather = (uint32_t)warp_sum(n_gather);
    if (lane == 0) {
        a.counts[q] = total;
        a.status[q] = KMER_B200_QUERY_OK;
        if (heavy) atomicAdd(a.n_heavy, (unsigned long long)heavy);
        if (ACCOUNT && n_gather) atomicAdd(a.gather_count, (unsigned long long)n_gather);
    }
}

// copy the in-record windows among the bucket entries from lo on into out[0..c) (seed offset j), one lane
template <bool COLL, bool ACCOUNT>
__device__ __forceinline__ void copy_lane(const SeedArgs &a, const Element &E, uint64_t lo, uint64_t c, uint64_t out, uint32_t j,
                                          uint32_t *n_gather) {
    for (uint64_t t = 0, w = 0; w < c; ++t) {
        const uint32_t p = gather32(pos_ptr(E, lo + t));
        if (ACCOUNT) *n_gather += ((lo + t) % 8 == 0 || t == 0) ? 1 : 0;
        if (COLL) {
            if (ACCOUNT) ++*n_gather;
            if (!window_in_record(a.index->boundary, p, a.k)) continue;
        }
        a.positions[out + w] = p;
        a.seed_offsets[out + w] = j;
        ++w;
    }
}

// the same with the whole warp (every lane passes the same arguments); UNROLL entries per lane and round in flight
template <bool COLL, bool ACCOUNT, int UNROLL>
__device__ __forceinline__ void copy_warp(const SeedArgs &a, const Element &E, uint64_t lo, uint64_t c, uint64_t out, uint32_t j,
                                          int lane, uint32_t *n_gather) {
    if (!COLL) {
        for (uint64_t t0 = 0; t0 < c; t0 += 32 * UNROLL) {
            uint32_t p[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const uint64_t t = t0 + u * 32 + lane;
                if (t < c) p[u] = gather32(pos_ptr(E, lo + t));
            }
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const uint64_t t = t0 + u * 32 + lane;
                if (t < c) {
                    a.positions[out + t] = p[u];
                    a.seed_offsets[out + t] = j;
                    if (ACCOUNT && ((lo + t) % 8 == 0 || t == 0)) ++*n_gather;
                }
            }
        }
        return;
    }
    const uint32_t lt = (1u << lane) - 1;
    for (uint64_t t0 = 0, w = 0; w < c; t0 += 32) {
        // the bucket holds at least c in-record entries from lo on: whatever this round reads behind it lands at o >= c
        const uint64_t t = t0 + lane;
        bool ok = false;
        uint32_t p = 0;
        if (lo + t < E.n_kmers) {
            p = gather32(pos_ptr(E, lo + t));
            ok = window_in_record(a.index->boundary, p, a.k);
            if (ACCOUNT) *n_gather += 1 + (((lo + t) % 8 == 0 || t == 0) ? 1 : 0);
        }
        const uint32_t b = __ballot_sync(kFull, ok);
        const uint64_t o = w + __popc(b & lt);
        if (ok && o < c) {
            a.positions[out + o] = p;
            a.seed_offsets[out + o] = j;
        }
        w += __popc(b);
    }
}

template <bool COLL, bool ACCOUNT>
__global__ void __launch_bounds__(kSeedThreads) seed_write_kernel(const SeedArgs a) {
    const int lane = threadIdx.x & 31;
    const uint64_t q = (uint64_t)blockIdx.x * kSeedWarps + threadIdx.x / 32;
    if (q >= a.n_queries) return;
    uint64_t out = a.counts[q];
    if (a.counts[q + 1] == out) return;
    const Element &E = a.index->elem[a.elem];
    const uint64_t i0 = a.kmer_base[q], i1 = a.kmer_base[q + 1];
    const uint64_t cap = a.max_occ ? (uint64_t)a.max_occ : ~0ull;
    uint32_t n_gather = 0;
    for (uint64_t r0 = i0; r0 < i1; r0 += 32) {
        const uint64_t i = r0 + lane;
        uint64_t c = 0, lo = 0;
        if (i < i1) {
            c = a.kmer_counts[i];
            if (c > cap) c = 0;
            if (c) lo = a.bucket_lo[i];
        }
        const uint64_t incl = warp_scan(c, lane);
        const uint64_t o = out + incl - c;
        const uint32_t j = (uint32_t)(i - i0);
        if (c > kHeavyCandidates) {
            const unsigned long long slot = atomicAdd(a.n_heavy, 1ull);
            a.heavy[slot] = HeavySeed{o, c, (uint32_t)lo, j};
        } else if (c && c <= kSeedLaneCopy) {
            copy_lane<COLL, ACCOUNT>(a, E, lo, c, o, j, &n_gather);
        }
        uint32_t todo = __ballot_sync(kFull, c > kSeedLaneCopy && c <= kHeavyCandidates);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            copy_warp<COLL, ACCOUNT, 1>(a, E, __shfl_sync(kFull, lo, src), __shfl_sync(kFull, c, src), __shfl_sync(kFull, o, src),
                                        __shfl_sync(kFull, j, src), lane, &n_gather);
        }
        out += __shfl_sync(kFull, incl, 31);
    }
    if (ACCOUNT) {
        n_gather = (uint32_t)warp_sum(n_gather);
        if (lane == 0 && n_gather) atomicAdd(a.gather_count, (unsigned long long)n_gather);
    }
}

// one warp per heavy bucket of the write pass
template <bool COLL, bool ACCOUNT>
__global__ void __launch_bounds__(kSeedThreads) seed_heavy_kernel(const SeedArgs a) {
    const int lane = threadIdx.x & 31;
    const Element &E = a.index->elem[a.elem];
    const uint64_t n = *a.n_heavy;
    uint32_t n_gather = 0;
    for (uint64_t h = (uint64_t)blockIdx.x * kSeedWarps + threadIdx.x / 32; h < n; h += (uint64_t)gridDim.x * kSeedWarps) {
        const HeavySeed s = a.heavy[h];
        copy_warp<COLL, ACCOUNT, 4>(a, E, s.lo, s.cnt, s.out, s.j, lane, &n_gather);
    }
    if (ACCOUNT) {
        n_gather = (uint32_t)warp_sum(n_gather);
        if (lane == 0 && n_gather) atomicAdd(a.gather_count, (unsigned long long)n_gather);
    }
}

__global__ void __launch_bounds__(256) seed_kmers_per_query_kernel(const uint64_t *__restrict__ q_offsets, uint64_t n_queries, uint32_t k,
                                                                   uint64_t *__restrict__ n_kmers) {
    for (uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_queries; q += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t m = q_offsets[q + 1] - q_offsets[q];
        n_kmers[q] = m >= k ? m - k + 1 : 0;
    }
}

template <bool COLL, bool ACCOUNT>
void launch_seed_pass(const SeedArgs &a, bool write, cudaStream_t stream) {
    const unsigned blocks = (unsigned)((a.n_queries + kSeedWarps - 1) / kSeedWarps);
    if (!write) {
        seed_count_kernel<COLL, ACCOUNT><<<blocks, kSeedThreads, 0, stream>>>(a);
        return;
    }
    seed_write_kernel<COLL, ACCOUNT><<<blocks, kSeedThreads, 0, stream>>>(a);
    if (a.heavy) seed_heavy_kernel<COLL, ACCOUNT><<<device_sm_count() * 2, kSeedThreads, 0, stream>>>(a);
}

}  // namespace

void launch_seed_kmers_per_query(const uint64_t *d_q_offsets, uint64_t n_queries, uint32_t k, uint64_t *d_n_kmers, cudaStream_t stream) {
    if (n_queries == 0) return;
    const uint64_t blocks = std::min<uint64_t>((n_queries + 255) / 256, (uint64_t)device_sm_count() * 8);
    seed_kmers_per_query_kernel<<<(unsigned)blocks, 256, 0, stream>>>(d_q_offsets, n_queries, k, d_n_kmers);
}

void launch_seed_count(const SeedArgs &a, cudaStream_t stream) {
    if (a.n_queries == 0) return;
    if (a.coll) a.gather_count ? launch_seed_pass<true, true>(a, false, stream) : launch_seed_pass<true, false>(a, false, stream);
    else a.gather_count ? launch_seed_pass<false, true>(a, false, stream) : launch_seed_pass<false, false>(a, false, stream);
}

void launch_seed_write(const SeedArgs &a, cudaStream_t stream) {
    if (a.n_queries == 0) return;
    if (a.coll) a.gather_count ? launch_seed_pass<true, true>(a, true, stream) : launch_seed_pass<true, false>(a, true, stream);
    else a.gather_count ? launch_seed_pass<false, true>(a, true, stream) : launch_seed_pass<false, false>(a, true, stream);
}

}  // namespace kb
