// Record votes of a read batch on a collection index (sm_100a): for each read q and each record r, votes(q, r) = the number
// of counted k-mers of q (1 <= in-record occurrences, <= max_occ when a cap is set) that occur in r; per read every
// (r, votes) with votes >= min_votes, by votes descending, then record ascending.
//
// One warp per read walks its k-mers like seed_count_kernel: tiles of kVoteTileSymbols symbols packed into shared memory
// by pack_query_group, one k-mer per lane and round, looked up with bucket_of; the in-record occurrences of a bucket are
// walked by the k-mer's own lane (short buckets) or by the whole warp (long ones). Each occurrence p is mapped to its record
// by a binary search over the record starts (the rule of locate_kernel). A bucket ascends in position, so its records do
// not decrease: an occurrence's record is new for the k-mer exactly when it differs from the previous in-record
// occurrence's record, and each new record is one vote. Votes go into a per-warp open-addressing table in shared memory.
//
// Count pass (votes_count_kernel): kmer_counts / bucket_lo per k-mer as seeding keeps them (so later passes neither pack,
// hash nor look up again), kmer_hits[q], n_pairs[q] = the new (k-mer, record) events of the read, and counts[q] = the
// table's entries with votes >= min_votes. A read whose distinct records exceed kVoteCapacity is flagged (ovf[q] = 1) and
// its counts[q] is left to the overflow path.
// Write pass (votes_walk_kernel<false>): an unflagged read rebuilds its table from the buckets, compacts the survivors and
// writes each one at its rank in (votes desc, record asc) order.
// Overflow path: votes_walk_kernel<true> writes the flagged read's new records to its segment of a global scratch array
// (segments sized by n_pairs), launch_segment_sort orders each segment, votes_runs_kernel run-length counts it and keeps the
// runs with votes >= min_votes (record order), and votes_place_kernel + two stable pair sorts (by votes descending, then by
// read) + votes_scatter_kernel put them at the read's offsets in (votes desc, record asc) order.
#include <algorithm>

#include "launch.h"
#include "query_pack.cuh"

namespace kb {

namespace {

constexpr int kVoteThreads = 256;
constexpr int kVoteWarps = kVoteThreads / 32;
constexpr uint32_t kVoteTileSymbols = 256;                   // one round of pack_query_group<32>: 8 symbols per lane
constexpr uint32_t kVoteTileWords = kVoteTileSymbols / 8 + 2;  // 8-bit symbols + the two zero words
constexpr uint32_t kLogSlots = 9;
constexpr uint32_t kSlots = 1u << kLogSlots;                  // per warp: 512 x (record, votes) = 4 KB
constexpr uint32_t kEmpty = 0xFFFFFFFFu;
constexpr uint32_t kLaneWalk = 4;                             // later passes: k-mers of up to this many occurrences per lane
constexpr uint32_t kFull = 0xFFFFFFFFu;

__device__ __forceinline__ uint64_t warp_sum(uint64_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// the last r with starts[r] <= p (p inside the text)
__device__ __forceinline__ uint32_t record_of(const VoteArgs &a, uint64_t p) {
    uint64_t lo = 0, hi = a.n_records;
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (__ldg(a.starts + mid) <= p) lo = mid;
        else hi = mid;
    }
    return (uint32_t)lo;
}

// one warp's table: keys kEmpty = free; *ovf set once more than kVoteCapacity records have been claimed (or a probe found
// no slot), after which nothing is added
struct VoteTable {
    uint32_t *key, *val, *used, *ovf;
    __device__ __forceinline__ void add(uint32_t r) const {
        if (*(volatile uint32_t *)ovf) return;
        uint32_t h = (r * 0x9E3779B1u) >> (32 - kLogSlots);
        for (uint32_t i = 0; i < kSlots; ++i, h = (h + 1) & (kSlots - 1)) {
            uint32_t k = ((volatile uint32_t *)key)[h];
            if (k == kEmpty) {
                k = atomicCAS(key + h, kEmpty, r);
                if (k == kEmpty) {
                    atomicAdd(val + h, 1u);
                    if (atomicAdd(used, 1u) >= kVoteCapacity) *(volatile uint32_t *)ovf = 1;
                    return;
                }
            }
            if (k == r) {
                atomicAdd(val + h, 1u);
                return;
            }
        }
        *(volatile uint32_t *)ovf = 1;
    }
};

// a flagged read's segment of the overflow scratch: every new record appended (order does not matter, it is sorted)
struct VoteSpill {
    uint32_t *out, *n;
    __device__ __forceinline__ void add(uint32_t r) const { out[atomicAdd(n, 1u)] = r; }
};

// The in-record occurrences among the bucket entries [lo, lo + cnt), counted up to `stop`, by one lane. VOTE: each one's
// record is added to `sink` when it differs from the previous one's (n_new counts those).
template <bool VOTE, typename Sink>
__device__ __forceinline__ uint64_t walk_lane(const VoteArgs &a, const Element &E, uint64_t lo, uint64_t cnt, uint64_t stop,
                                              const Sink &sink, uint32_t *n_new) {
    const uint64_t *boundary = a.index->boundary;
    uint64_t c = 0;
    uint32_t prev = kEmpty;
    for (uint64_t t = 0; t < cnt && c < stop; ++t) {
        const uint32_t p = gather32(pos_ptr(E, lo + t));
        if (!window_in_record(boundary, p, a.k)) continue;
        ++c;
        if (VOTE) {
            const uint32_t r = record_of(a, p);
            if (r != prev) {
                prev = r;
                ++*n_new;
                sink.add(r);
            }
        }
    }
    return c;
}

// the same with the whole warp, 32 entries per round (every lane passes the same lo, cnt, stop); only the first `stop`
// in-record occurrences vote
template <bool VOTE, typename Sink>
__device__ __forceinline__ uint64_t walk_warp(const VoteArgs &a, const Element &E, uint64_t lo, uint64_t cnt, uint64_t stop,
                                              int lane, const Sink &sink, uint32_t *n_new) {
    const uint64_t *boundary = a.index->boundary;
    const uint32_t lt = (1u << lane) - 1;
    uint64_t c = 0;
    uint32_t prev = kEmpty;  // the record of the last in-record occurrence of the rounds before
    for (uint64_t t0 = 0; t0 < cnt && c < stop; t0 += 32) {
        const uint64_t t = t0 + lane;
        bool ok = false;
        uint32_t p = 0;
        if (t < cnt) {
            p = gather32(pos_ptr(E, lo + t));
            ok = window_in_record(boundary, p, a.k);
        }
        const uint32_t b = __ballot_sync(kFull, ok);
        if (VOTE) {
            ok = ok && c + __popc(b & lt) < stop;
            const uint32_t r = ok ? record_of(a, p) : 0;
            const uint32_t v = __ballot_sync(kFull, ok);
            const uint32_t below = v & lt;
            const uint32_t r_below = __shfl_sync(kFull, r, below ? 31 - __clz(below) : lane);
            if (ok && r != (below ? r_below : prev)) {
                ++*n_new;
                sink.add(r);
            }
            if (v) prev = __shfl_sync(kFull, r, 31 - __clz(v));
        }
        c += __popc(b);
    }
    return min(c, stop);
}

struct NoSink {
    __device__ __forceinline__ void add(uint32_t) const {}
};

__device__ __forceinline__ void table_clear(uint32_t *key, uint32_t *val, int lane) {
    for (uint32_t s = lane; s < kSlots; s += 32) {
        key[s] = kEmpty;
        val[s] = 0;
    }
}

__global__ void __launch_bounds__(kVoteThreads) votes_count_kernel(const VoteArgs a) {
    __shared__ uint64_t smem_q[kVoteWarps][kVoteTileWords];
    __shared__ uint32_t smem_key[kVoteWarps][kSlots], smem_val[kVoteWarps][kSlots];
    __shared__ uint32_t smem_used[kVoteWarps], smem_ovf[kVoteWarps];
    const int lane = threadIdx.x & 31, w = threadIdx.x / 32;
    const uint64_t q = (uint64_t)blockIdx.x * kVoteWarps + w;
    if (q >= a.n_queries) return;
    const DeviceIndex &ix = *a.index;
    const PackedText T = ix.text;
    const Element &E = ix.elem[a.elem];
    uint64_t *qw = smem_q[w];
    const VoteTable tab{smem_key[w], smem_val[w], &smem_used[w], &smem_ovf[w]};
    table_clear(tab.key, tab.val, lane);
    if (lane == 0) smem_used[w] = smem_ovf[w] = 0;
    __syncwarp();
    const uint64_t off0 = a.q_offsets[q];
    const uint64_t m = a.q_offsets[q + 1] - off0;
    const uint64_t i0 = a.kmer_base[q];
    const uint32_t k = a.k;
    const uint64_t cap = a.max_occ ? (uint64_t)a.max_occ : ~0ull;
    const uint64_t stop = a.max_occ ? (uint64_t)a.max_occ + 1 : ~0ull;  // a count above max_occ is kept as max_occ + 1
    const uint32_t step = kVoteTileSymbols - (k - 1);
    uint32_t hits = 0, n_new = 0;
    for (uint64_t j0 = 0; j0 < m; j0 += step) {
        const uint32_t ts = (uint32_t)min((uint64_t)kVoteTileSymbols, m - j0);
        pack_query_group<32>(a.q_ranks, off0 + j0, ts, a.q_offsets[a.n_queries], T, (uint32_t)lane, kFull, a.error_flag, qw);
        const uint32_t nk = ts >= k ? ts - k + 1 : 0;
        for (uint32_t t0 = 0; t0 < nk; t0 += 32) {
            const uint32_t t = t0 + lane;
            Range r{0, 0};
            if (t < nk) r = bucket_of(E, key_at(qw, (uint64_t)t, k, T.bits, T.sigma));
            // without a cap every occurrence votes on the first walk; with one, a k-mer votes on a second walk once its
            // count is known to be <= max_occ
            uint64_t c = 0;
            const bool big = r.cnt > 32;
            if (!big) c = a.max_occ ? walk_lane<false>(a, E, r.lo, r.cnt, stop, NoSink{}, &n_new)
                                    : walk_lane<true>(a, E, r.lo, r.cnt, stop, tab, &n_new);
            uint32_t todo = __ballot_sync(kFull, big);
            while (todo) {
                const int src = __ffs(todo) - 1;
                todo &= todo - 1;
                const uint64_t lo = __shfl_sync(kFull, r.lo, src), cnt = __shfl_sync(kFull, r.cnt, src);
                const uint64_t cw = a.max_occ ? walk_warp<false>(a, E, lo, cnt, stop, lane, NoSink{}, &n_new)
                                              : walk_warp<true>(a, E, lo, cnt, stop, lane, tab, &n_new);
                if (lane == src) c = cw;
            }
            const bool counted = c >= 1 && c <= cap;
            if (a.max_occ) {
                if (counted && !big) walk_lane<true>(a, E, r.lo, r.cnt, c, tab, &n_new);
                todo = __ballot_sync(kFull, counted && big);
                while (todo) {
                    const int src = __ffs(todo) - 1;
                    todo &= todo - 1;
                    walk_warp<true>(a, E, __shfl_sync(kFull, r.lo, src), __shfl_sync(kFull, r.cnt, src), __shfl_sync(kFull, c, src),
                                    lane, tab, &n_new);
                }
            }
            if (t < nk) {
                const uint64_t i = i0 + j0 + t;
                a.kmer_counts[i] = (uint32_t)min(c, stop);
                a.bucket_lo[i] = (uint32_t)r.lo;
                hits += counted ? 1 : 0;
            }
        }
        __syncwarp();  // the tile is read by every lane before the next one is packed over it
        if (j0 + ts >= m) break;
    }
    hits = (uint32_t)warp_sum(hits);
    n_new = (uint32_t)warp_sum(n_new);
    const bool ovf = smem_ovf[w] != 0;
    uint32_t kept = 0;
    if (!ovf)
        for (uint32_t s = lane; s < kSlots; s += 32) kept += (tab.key[s] != kEmpty && tab.val[s] >= a.min_votes) ? 1 : 0;
    kept = (uint32_t)warp_sum(kept);
    if (lane == 0) {
        a.counts[q] = kept;
        a.kmer_hits[q] = hits;
        a.n_pairs[q] = ovf ? n_new : 0;
        a.ovf[q] = ovf ? 1 : 0;
        a.status[q] = KMER_B200_QUERY_OK;
        if (ovf) atomicAdd(a.n_ovf, 1ull);
    }
}

// Later passes: the warp walks the counted k-mers of read q again from kmer_counts / bucket_lo and adds their records to
// `sink`. The bucket holds at least c in-record entries from lo on, so the walks stop inside it.
template <typename Sink>
__device__ __forceinline__ void rewalk(const VoteArgs &a, const Element &E, uint64_t q, int lane, const Sink &sink) {
    const uint64_t i0 = a.kmer_base[q], i1 = a.kmer_base[q + 1];
    const uint64_t cap = a.max_occ ? (uint64_t)a.max_occ : ~0ull;
    uint32_t n_new = 0;
    for (uint64_t r0 = i0; r0 < i1; r0 += 32) {
        const uint64_t i = r0 + lane;
        uint64_t c = 0, lo = 0;
        if (i < i1) {
            c = a.kmer_counts[i];
            if (c > cap) c = 0;
            if (c) lo = a.bucket_lo[i];
        }
        if (c && c <= kLaneWalk) walk_lane<true>(a, E, lo, E.n_kmers - lo, c, sink, &n_new);
        uint32_t todo = __ballot_sync(kFull, c > kLaneWalk);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const uint64_t l = __shfl_sync(kFull, lo, src);
            walk_warp<true>(a, E, l, E.n_kmers - l, __shfl_sync(kFull, c, src), lane, sink, &n_new);
        }
    }
}

// SPILL = false: the write pass of the unflagged reads; SPILL = true: the flagged reads' records to their scratch segments
template <bool SPILL>
__global__ void __launch_bounds__(kVoteThreads, 1) votes_walk_kernel(const VoteArgs a) {
    __shared__ uint32_t smem_key[SPILL ? 1 : kVoteWarps][kSlots], smem_val[SPILL ? 1 : kVoteWarps][kSlots];
    __shared__ uint32_t smem_used[kVoteWarps], smem_ovf[kVoteWarps];
    const int lane = threadIdx.x & 31, w = threadIdx.x / 32;
    const uint64_t q = (uint64_t)blockIdx.x * kVoteWarps + w;
    if (q >= a.n_queries || (a.ovf[q] != 0) != SPILL) return;
    const Element &E = a.index->elem[a.elem];
    if (SPILL) {
        if (lane == 0) smem_used[w] = 0;
        __syncwarp();
        rewalk(a, E, q, lane, VoteSpill{a.spill + a.spill_off[q], &smem_used[w]});
        return;
    }
    uint64_t out = a.counts[q];
    const uint32_t n_out = (uint32_t)(a.counts[q + 1] - out);
    if (n_out == 0) return;
    uint32_t *key = smem_key[SPILL ? 0 : w], *val = smem_val[SPILL ? 0 : w];
    table_clear(key, val, lane);
    if (lane == 0) smem_used[w] = smem_ovf[w] = 0;
    __syncwarp();
    rewalk(a, E, q, lane, VoteTable{key, val, &smem_used[w], &smem_ovf[w]});
    __syncwarp();
    // the survivors to the front of the table, in slot order (a slot is read before any lane writes at or below it)
    const uint32_t lt = (1u << lane) - 1;
    uint32_t n = 0;
    for (uint32_t s0 = 0; s0 < kSlots; s0 += 32) {
        const uint32_t kk = key[s0 + lane], vv = val[s0 + lane];
        const bool keep = kk != kEmpty && vv >= a.min_votes;
        const uint32_t b = __ballot_sync(kFull, keep);
        if (keep) {
            key[n + __popc(b & lt)] = kk;
            val[n + __popc(b & lt)] = vv;
        }
        n += __popc(b);
        __syncwarp();
    }
    // rank of each survivor in (votes desc, record asc) order
    for (uint32_t i = lane; i < n; i += 32) {
        const uint32_t ri = key[i], vi = val[i];
        uint32_t rank = 0;
        for (uint32_t j = 0; j < n; ++j) {
            const uint32_t rj = key[j], vj = val[j];
            rank += (vj > vi || (vj == vi && rj < ri)) ? 1 : 0;
        }
        a.records[out + rank] = ri;
        a.votes[out + rank] = vi;
    }
}

// a flagged read's sorted segment -> its runs (record, length) with length >= min_votes, in record order, at the front of
// the segment in run_records / run_votes; counts[q] and flagged[q] = their number
__global__ void __launch_bounds__(kVoteThreads) votes_runs_kernel(const VoteArgs a, uint32_t *run_records, uint32_t *run_votes,
                                                                   uint64_t *flagged) {
    const int lane = threadIdx.x & 31;
    const uint64_t q = (uint64_t)blockIdx.x * kVoteWarps + threadIdx.x / 32;
    if (q >= a.n_queries || !a.ovf[q]) return;
    const uint64_t s0 = a.spill_off[q], s1 = a.spill_off[q + 1];
    const uint32_t *x = a.spill;
    const uint32_t lt = (1u << lane) - 1, le = lt | (1u << lane);
    uint64_t run_start = s0, out = s0;
    for (uint64_t base = s0; base < s1; base += 32) {
        const uint64_t s = base + lane;
        const bool valid = s < s1;
        const uint32_t v = valid ? x[s] : 0;
        const bool is_start = valid && (s == s0 || x[s - 1] != v);
        const bool is_end = valid && (s + 1 == s1 || x[s + 1] != v);
        const uint32_t starts = __ballot_sync(kFull, is_start);
        const uint32_t below = starts & le;
        const uint64_t my_start = below ? base + 31 - __clz(below) : run_start;
        const uint64_t votes = s - my_start + 1;
        const bool keep = is_end && votes >= a.min_votes;
        const uint32_t kb = __ballot_sync(kFull, keep);
        if (keep) {
            run_records[out + __popc(kb & lt)] = v;
            run_votes[out + __popc(kb & lt)] = (uint32_t)votes;
        }
        out += __popc(kb);
        if (starts) run_start = base + 31 - __clz(starts);
    }
    if (lane == 0) a.counts[q] = flagged[q] = out - s0;
}

// the flagged reads' runs as one list: entry c = flagged_off[q] + i (run i of read q), sort key ~votes, value c
__global__ void __launch_bounds__(kVoteThreads) votes_place_kernel(const VoteArgs a, const uint32_t *run_records,
                                                                    const uint32_t *run_votes, const uint64_t *flagged_off,
                                                                    uint32_t *keys, uint32_t *vals, uint32_t *c_rec,
                                                                    uint32_t *c_votes, uint32_t *c_read) {
    const int lane = threadIdx.x & 31;
    const uint64_t q = (uint64_t)blockIdx.x * kVoteWarps + threadIdx.x / 32;
    if (q >= a.n_queries || !a.ovf[q]) return;
    const uint64_t s0 = a.spill_off[q], c0 = flagged_off[q], n = flagged_off[q + 1] - c0;
    for (uint64_t i = lane; i < n; i += 32) {
        const uint64_t c = c0 + i;
        keys[c] = ~run_votes[s0 + i];
        vals[c] = (uint32_t)c;
        c_rec[c] = run_records[s0 + i];
        c_votes[c] = run_votes[s0 + i];
        c_read[c] = (uint32_t)q;
    }
}

__global__ void __launch_bounds__(256) votes_owner_kernel(const uint32_t *vals, const uint32_t *c_read, uint64_t n, uint32_t *keys) {
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (uint64_t)gridDim.x * blockDim.x)
        keys[c] = c_read[vals[c]];
}

// after the sorts by votes descending and then by read: entry c of the list is rank c - flagged_off[q] of its read q
__global__ void __launch_bounds__(256) votes_scatter_kernel(const VoteArgs a, const uint32_t *vals, const uint32_t *c_rec,
                                                            const uint32_t *c_votes, const uint32_t *c_read,
                                                            const uint64_t *flagged_off, uint64_t n) {
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t s = vals[c];
        const uint32_t q = c_read[s];
        const uint64_t o = a.counts[q] + (c - flagged_off[q]);
        a.records[o] = c_rec[s];
        a.votes[o] = c_votes[s];
    }
}

unsigned warps_grid(uint64_t n_queries) { return (unsigned)((n_queries + kVoteWarps - 1) / kVoteWarps); }
unsigned flat_grid(uint64_t n) { return (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)device_sm_count() * 8); }

}  // namespace

void launch_votes_count(const VoteArgs &a, cudaStream_t stream) {
    if (a.n_queries) votes_count_kernel<<<warps_grid(a.n_queries), kVoteThreads, 0, stream>>>(a);
}

void launch_votes_write(const VoteArgs &a, cudaStream_t stream) {
    if (a.n_queries) votes_walk_kernel<false><<<warps_grid(a.n_queries), kVoteThreads, 0, stream>>>(a);
}

void launch_votes_spill(const VoteArgs &a, uint32_t *run_records, uint32_t *run_votes, uint64_t *flagged, cudaStream_t stream) {
    if (a.n_queries == 0) return;
    votes_walk_kernel<true><<<warps_grid(a.n_queries), kVoteThreads, 0, stream>>>(a);
    launch_segment_sort(a.spill, run_records, a.spill_off, a.ovf, a.n_queries, a.record_bits, stream);
    votes_runs_kernel<<<warps_grid(a.n_queries), kVoteThreads, 0, stream>>>(a, run_records, run_votes, flagged);
}

void launch_votes_place(const VoteArgs &a, const uint32_t *run_records, const uint32_t *run_votes, const uint64_t *flagged_off,
                        uint32_t *keys, uint32_t *vals, uint32_t *c_rec, uint32_t *c_votes, uint32_t *c_read, cudaStream_t stream) {
    if (a.n_queries)
        votes_place_kernel<<<warps_grid(a.n_queries), kVoteThreads, 0, stream>>>(a, run_records, run_votes, flagged_off, keys, vals,
                                                                                  c_rec, c_votes, c_read);
}

void launch_votes_owner(const uint32_t *vals, const uint32_t *c_read, uint64_t n, uint32_t *keys, cudaStream_t stream) {
    if (n) votes_owner_kernel<<<flat_grid(n), 256, 0, stream>>>(vals, c_read, n, keys);
}

void launch_votes_scatter(const VoteArgs &a, const uint32_t *vals, const uint32_t *c_rec, const uint32_t *c_votes, const uint32_t *c_read,
                          const uint64_t *flagged_off, uint64_t n, cudaStream_t stream) {
    if (n) votes_scatter_kernel<<<flat_grid(n), 256, 0, stream>>>(a, vals, c_rec, c_votes, c_read, flagged_off, n);
}

}  // namespace kb
