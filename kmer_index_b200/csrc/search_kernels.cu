// Batched search kernels (sm_100a): the replacement for kmer_index::search (kmer_index.hpp:505-558),
// kmer_index_element::search (kmer_index.hpp:193-346) and kmer_index_result::to_vector
// (kmer_index_result.hpp:244-260).
//
// A group of G lanes per query (G = 1, 2, 4, 8 or 32, chosen per batch). The group
//   1. packs the query into shared memory (same b-bit MSB-first layout as the text),
//   2. derives the query's plan from its length and the scheme table (which element(s), which parts),
//   3. looks the parts it needs up in the directory (one lane per part) -- one loop for every plan; the
//      reference's early "part absent => empty result" return and its throw for short rests are decided
//      here, in the reference's order,
//   4. walks the seed bucket G candidates at a time; every lane checks its candidate's remaining
//      constraints, a list of (text offset, query offset, length) spans, directly against the packed text
//      (the text is the intersection oracle: position x is in bucket hash(T[x,x+k)) and in no other, so
//      "p + d is in the bucket of part j" is "T[p+d, p+d+k) == part j"); hits are compacted with ballot/popc.
// Results are produced in two passes (count -> exclusive scan -> write) so the output is an exact CSR; the count
// pass lists the queries that have hits and the write pass visits only those.
#include <algorithm>

#include "radix.cuh"
#include "launch.h"
#include "query_pack.cuh"

namespace kb {

constexpr int kSearchWarps = 8;
constexpr int kSearchThreads = kSearchWarps * 32;
#ifndef KB_SEARCH_MIN_BLOCKS
#define KB_SEARCH_MIN_BLOCKS 8  // <= 32 registers: 2048 threads per SM in flight beats the few spills (profiles/)
#endif

enum PlanKind : int { kExact = 0, kSubK = 1, kContig = 2, kBuggySingle = 3, kMultiSum = 4 };

// One group of G lanes per query (one lane up to 64 symbols ... a full warp for long queries or long buckets): the scalar part
// of a query (plan, status) costs a warp instruction per group, not per warp, and G/32 more queries are in
// flight per SM to cover the chain of dependent gathers (offsets -> ranks -> directory -> bucket -> text).
// Candidate lists longer than this are not walked by a small group: the query is appended to the batch's
// "heavy" list and a second launch gives it a full warp (long buckets of repetitive / low-entropy text): kHeavyCandidates.

// HEAVY = true: the second launch (G = 32) over the heavy list; never hands a query off again.
// VIEWS = true: elements may be prefix views of the largest k's arrays (shared-positions index, Element::width); compiled
// only into the warp-per-query kernels below (search_views_kernel), so the ordinary variants pay nothing for it.
template <int PASS_, int G, bool HEAVY, bool SINGLE, bool VIEWS = false>
__device__ __forceinline__ void search_query(const SearchArgs &a, const uint64_t q, uint64_t *smem_q) {
    // count pass variants: + sum of the gathered sectors; + whole-text rule left for the epilogue (sharded)
    constexpr bool kAccount = PASS_ == kPassCountAccount || PASS_ == kPassCountDeferredAccount;
    constexpr bool kDefer = PASS_ == kPassCountDeferred || PASS_ == kPassCountDeferredAccount;
    constexpr int PASS = (kAccount || kDefer) ? (int)kPassCount : PASS_;
    const int lane = threadIdx.x & 31;
    const int gl = threadIdx.x & (G - 1);          // lane inside the group
    const int group = threadIdx.x / G;             // group inside the CTA
    const uint32_t gshift = (uint32_t)(lane - gl);  // first warp lane of the group
    const uint32_t gfull = G == 32 ? 0xFFFFFFFFu : ((1u << G) - 1);
    const uint32_t gmask = gfull << gshift;
    const uint32_t lt_mask = (1u << gl) - 1;
// a group of one lane needs no warp collectives: they fold to the lane's own value at compile time
#define GBALLOT(pred) (G == 1 ? ((pred) ? 1u : 0u) : ((__ballot_sync(gmask, (pred)) >> gshift) & gfull))
#define GSHFL(v, src) (G == 1 ? (v) : __shfl_sync(gmask, (v), (src), G))
// hand the query to the heavy launch: the count pass enlists it (and reports no hits for now) and marks it in
// unsorted[q] bit 1; the write pass follows that mark (below), never its own candidate count -- the two can differ
// once an auxiliary element has been built between the passes
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
        if (a.counts[q + 1] == out_base) return;  // nothing to write (also covers every non-OK status)
        if (!HEAVY && G < 32 && (a.unsorted[q] & 2)) return;  // the count pass gave it to the heavy launch (which only follows
                                                             // a pass of narrower groups: a full-warp pass writes it itself)
    }

    const DeviceIndex &ix = *a.index;
    const PackedText T = ix.text;
    uint64_t *qw = smem_q + (size_t)group * a.q_words;
    const bool packed_in = a.q_packed != nullptr;
    const uint64_t off0 = packed_in ? 0 : a.q_offsets[q];
    const uint64_t m64 = packed_in ? (uint64_t)a.q_lens16[q] : a.q_offsets[q + 1] - off0;
    const uint64_t q_total = packed_in ? 0 : a.q_offsets[a.n_queries];  // symbols in q_ranks: bounds the 16-byte reads

    uint32_t status = KMER_B200_QUERY_OK;
    if (m64 == 0) {
        status = KMER_B200_QUERY_UNDEFINED;  // assert(query.size() > 0), kmer_index.hpp:195
    } else if (a.mode == KMER_B200_MODE_REFERENCE_EXACT && m64 > kQuerySizeRange) {
        status = KMER_B200_QUERY_THROW_INVALID_ARGUMENT;  // kmer_index.hpp:507-509
    } else if (a.mode == KMER_B200_MODE_REFERENCE_EXACT && m64 == kQuerySizeRange) {
        status = KMER_B200_QUERY_UNDEFINED;  // out-of-bounds table read, kmer_index.hpp:512
    } else if (m64 > a.max_len) {
        status = KMER_B200_QUERY_TOO_LONG_FOR_SHARD;
    }
    if (status != KMER_B200_QUERY_OK) {
        if (gl == 0) {
            if (PASS == kPassCount) {
                a.counts[q] = 0;
                a.status[q] = (uint8_t)status;
                a.unsorted[q] = 0;
                if (kDefer) {
                    a.defer[q] = 0;
                    a.present4[q] = 0;
                }
            } else if (PASS == kPassPresence) {
                if (a.present4 != nullptr) a.present4[q] = 0; else a.present[q] = 0;
            }
        }
        return;
    }
    const uint32_t m = (uint32_t)m64;

    // ---- 1. pack the query (b bits per symbol, MSB-first) -----------------------------------------------
    if (packed_in) {
        // the caller packed the query already: copy its words (and the two zero words the window reads rely on)
        const uint32_t n_words = (m * T.bits + 63) / 64;
        const uint64_t *src = a.q_packed + q * a.q_stride;
        for (uint32_t w = gl; w < n_words; w += G) qw[w] = src[w];
        if (gl == 0) {
            qw[n_words] = 0;
            qw[n_words + 1] = 0;
        }
        if (G > 1) __syncwarp(gmask);
    } else {
        pack_query_group<G>(a.q_ranks, off0, m, q_total, T, (uint32_t)gl, gmask, a.error_flag, qw);
    }

    // ---- 2. plan -----------------------------------------------------------------------------------------
    int kind = kExact;
    uint32_t e0 = 0, k0 = 0, nparts = 1, P = 0, rest = 0;
    bool throw_after = false, from_list = false;
    const uint8_t *S = nullptr;
    if (a.mode == KMER_B200_MODE_CORRECT) {
        // any element answers correctly. Planner (SURVEY.md 8f.4, measured in profiles/r02/planner_report.md): the
        // smallest k >= m if there is one -- its bucket (k == m) or prefix slab (k > m) IS the result, n / sigma^m
        // positions and nothing to verify -- else the largest k, whose buckets are the shortest candidate lists
        // (n / sigma^k each) to verify against the text.
        if (!SINGLE) {
            e0 = ix.elem_by_k_desc[0];
            for (uint32_t i = ix.n_elems; i-- > 0;) {
                const uint32_t e = ix.elem_by_k_desc[i];
                if (ix.elem[e].k >= m) {
                    e0 = e;
                    break;
                }
            }
        }
        k0 = ix.elem[e0].k;
        kind = (m == k0) ? kExact : (m > k0 ? kContig : kSubK);
    } else {
        // single-k index: the table row is [k] for every length and the facade dispatches straight to the element
        // (kmer_index.hpp:512-513); SINGLE compiles the multi-k plans out (fewer live registers, fewer spills)
        uint32_t s_len = 1;
        bool multi = false;
        if (SINGLE) {
            e0 = 0;
            k0 = ix.elem[0].k;
        } else {
            const uint32_t s_off = ix.scheme.sum_off[m];
            s_len = ix.scheme.sum_off[m + 1] - s_off;
            S = ix.scheme.sum_elem + s_off;
            e0 = S[0];
            k0 = ix.elem[e0].k;
            multi = ix.scheme.use_multi[m] && ix.n_elems > 1;  // kmer_index.hpp:512
        }
        if (!multi) {
            // kmer_index_element<k0>::search, kmer_index.hpp:193-346
            if (m == k0) {
                kind = kExact;
            } else if (m < k0) {
                if (ix.pow_sigma[k0 - m] > 10000000ull)  // kmer_index.hpp:119-122
                    status = KMER_B200_QUERY_THROW_INVALID_ARGUMENT;
                kind = kSubK;
            } else {
                P = m / k0;
                rest = m % k0;
                nparts = P;
                throw_after = rest > 0 && ix.pow_sigma[k0 - rest] > 10000000ull;  // :234 -> :119
                // :314 compares every later part against the LAST part when P >= 3 and rest > 0
                kind = (rest == 0 || P <= 2) ? kContig : kBuggySingle;
            }
        } else {
            // kmer_index.hpp:516-557
            from_list = true;
            nparts = s_len;
            kind = s_len == 1 ? kExact : (s_len == 2 ? kContig : kMultiSum);
        }
    }
    if (status != KMER_B200_QUERY_OK) {
        if (gl == 0) {
            if (PASS == kPassCount) {
                a.counts[q] = 0;
                a.status[q] = (uint8_t)status;
                a.unsorted[q] = 0;
                if (kDefer) {
                    a.defer[q] = 0;
                    a.present4[q] = 0;
                }
            } else if (PASS == kPassPresence) {
                if (a.present4 != nullptr) a.present4[q] = 0; else a.present[q] = 0;
            }
        }
        return;
    }

    bool was_subk = false;
    if (kind == kSubK) {
        if (m < 64 && ix.aux_for_len[m] != 0xFF) {  // an auxiliary k' = m element answers it as an exact lookup
            e0 = ix.aux_for_len[m];
            k0 = m;
            kind = kExact;
            nparts = 1;
            from_list = false;
            was_subk = true;  // no whole-text presence rule applies to prefix enumeration
        } else if (PASS == kPassCount && m < 64 && gl == 0) {
            atomicOr(reinterpret_cast<unsigned long long *>(a.error_flag + 2), 1ull << m);  // ask the host for one
        }
    }

    // algorithmic gathers of this lane (32-byte sectors at data-dependent addresses), summed per batch when asked
    uint32_t n_gather = 0;

    // ---- 3. presence of the indexed parts ------------------------------------------------------------------
    // The reference looks every indexed part up first and returns empty when one is absent (:216-227, :516-527).
    // Where the plan is a contiguous comparison of the whole query that rule is redundant -- an occurrence of
    // the query contains an occurrence of every part -- so the lookups are only done when the outcome depends on
    // them: the throw for short rests happens only if all parts are present, and the two defective plans do not
    // constrain every part's position.
    const bool need_presence = throw_after || kind == kBuggySingle || kind == kMultiSum;
    if (PASS == kPassPresence && (!need_presence || was_subk)) {  // nothing about this query depends on other shards
        if (gl == 0) {
            if (a.present4 != nullptr) a.present4[q] = 0; else a.present[q] = 0;
        }
        return;
    }
    Range seed{0, 0};       // candidate list: positions pos[seed.lo .. +cnt) of element seed_e, match start = pos - seed_d
    uint32_t seed_e = e0, seed_d = 0, seed_o = 0;  // ... and the seed part sits at query offset seed_o
    bool all_present = true;
    uint64_t present_mask = 0;
    // Every plan goes through the same lookup loop -- the lanes of a warp hold queries of different plans, and a
    // gather issued from one place is one round trip for all of them. A contiguous plan (or exact lookup) does one
    // lookup, part 0: any element finds the same occurrences, so it takes the element with the largest k <= m
    // (the shortest candidate list) and the rest of the query is compared against the text.
    uint32_t e_first = e0;
    if (!SINGLE && !need_presence && kind == kContig) {
        for (uint32_t i = 0; i < ix.n_elems; ++i) {
            const uint32_t e = ix.elem_by_k_desc[i];
            if (ix.elem[e].k <= m) {
                e_first = e;
                break;
            }
        }
    }
    const uint32_t n_lookups = need_presence ? nparts : 1;
    if (kind != kSubK) {
        uint64_t best_cnt = ~0ull;
        for (uint32_t base = 0; base < n_lookups; base += G) {
            const uint32_t j = base + gl;
            const bool valid = j < n_lookups;
            Range rg{0, 0};
            uint32_t e = e_first, o = j * k0, d = j * k0;
            bool foreign = false;
            uint32_t tail_slots = 0;  // views (Element::width): k-mer starts that are compared directly, and whether
            bool tail_hit = false;    // the part occurs at one of them
            if (valid) {
                if (from_list && need_presence) {  // `last_k = current_k` is not cumulative, kmer_index.hpp:526
                    e = S[j];
                    o = j ? ix.elem[S[j - 1]].k : 0;
                    d = j * ix.elem[S[0]].k;  // expected at text offset j * k_0 (:535,544)
                }
                const Element &E = ix.elem[e];
                const uint64_t key = key_at(qw, (uint64_t)o, E.k, T.bits, T.sigma);
                const uint64_t *pb = ix.presence[e];
                if (pb != nullptr && (key < E.key_lo || key >= E.key_hi)) {
                    // another part's hash (key-range multi-GPU search): whether it occurs anywhere in the text comes from
                    // the replicated presence bitmap; its positions live on another GPU, so it can never seed
                    foreign = true;
                    rg.cnt = ((gather64(pb + (key >> 6)) >> (key & 63)) & 1ull) ? 1 : 0;
                } else {
                    rg = bucket_of<VIEWS>(E, key);
                    if (VIEWS && E.width != 1) {
                        tail_slots = E.k_phys - E.k;
                        for (uint32_t t = 0; rg.cnt == 0 && !tail_hit && t < tail_slots; ++t)
                            tail_hit = match_span(T, qw, T.n - E.k_phys + 1 + t, o, E.k);
                    }
                }
                if (kAccount) n_gather += 1 + (E.shift ? 1 : 0);
            }
            const uint32_t here = GBALLOT(valid && (rg.cnt != 0 || tail_hit));
            if (base < 64) present_mask |= (uint64_t)here << base;
            const uint32_t want = GBALLOT(valid);
            if (need_presence && here != want) {
                all_present = false;
                // stop early only when the local answer is final (unsharded search)
                if (PASS != kPassPresence && !kDefer && a.present_global == nullptr && a.present_global4 == nullptr) break;
            }
            // seed from the shortest bucket among the parts whose position the plan constrains:
            // all of them, except the middle parts of the kmer_index.hpp:314 defect
            const bool seedable = valid && !foreign && (kind != kBuggySingle || j == 0 || j + 1 == nparts);
            uint64_t c = seedable ? rg.cnt + tail_slots : ~0ull;
            uint32_t who = gl;
            for (int off = G >> 1; off > 0; off >>= 1) {
                const uint64_t oc = __shfl_xor_sync(gmask, c, off, G);
                const uint32_t ow = __shfl_xor_sync(gmask, who, off, G);
                if (oc < c || (oc == c && ow < who)) {
                    c = oc;
                    who = ow;
                }
            }
            if (c < best_cnt) {
                best_cnt = c;
                seed.lo = GSHFL(rg.lo, who);
                seed.cnt = VIEWS ? GSHFL(rg.cnt, who) : c;
                seed_e = GSHFL(e, who);
                seed_d = GSHFL(d, who);
                if (VIEWS) seed_o = GSHFL(o, who);
            }
        }
    }
    if (PASS == kPassPresence) {
        if (gl == 0) {
            if (a.present4 != nullptr) {
                // one nibble per part so that a SUM all-reduce over <= 15 shards acts as an OR
                uint32_t enc = 0;
                for (uint32_t j = 0; j < 8; ++j) enc |= (uint32_t)((present_mask >> j) & 1) << (4 * j);
                a.present4[q] = enc;
            } else {
                a.present[q] = present_mask;
            }
        }
        return;
    }
    if (kDefer) {
        // publish this shard's flags and what the epilogue has to decide; the local absence of a part never
        // empties the result here (another shard may hold it), it only empties the local candidate list
        const bool rule = kind != kSubK && need_presence && !was_subk;
        if (gl == 0) {
            uint32_t enc = 0;
            if (rule)
                for (uint32_t j = 0; j < 8; ++j) enc |= (uint32_t)((present_mask >> j) & 1) << (4 * j);
            a.present4[q] = enc;
            // more than 8 parts cannot be encoded: parts = 63 makes the epilogue report no hits
            a.defer[q] = rule ? (uint8_t)(0x40u | (throw_after ? 0x80u : 0u) | (nparts <= 8 ? nparts : 63u)) : 0;
        }
        if (rule && throw_after) {  // either THROW or empty: no hits in both cases
            if (kAccount) {
                for (int o = G >> 1; o > 0; o >>= 1) n_gather += __shfl_xor_sync(gmask, n_gather, o, G);
                if (gl == 0) atomicAdd(a.gather_count, (unsigned long long)n_gather);
            }
            if (gl == 0) {
                a.counts[q] = 0;
                a.status[q] = KMER_B200_QUERY_OK;
                a.unsorted[q] = 0;
            }
            return;
        }
        all_present = true;
        throw_after = false;
    }
    if (!kDefer && kind != kSubK && need_presence && !was_subk) {
        // sharded: presence is a property of the whole text (kmer_index.hpp:216-227)
        if (a.present_global != nullptr) {
            const uint64_t full = nparts >= 64 ? ~0ull : ((1ull << nparts) - 1);
            all_present = (a.present_global[q] & full) == full;
        } else if (a.present_global4 != nullptr) {
            uint32_t x = a.present_global4[q];
            x = (x | (x >> 1) | (x >> 2) | (x >> 3)) & 0x11111111u;  // nibble j non-zero <=> part j occurs somewhere
            const uint32_t full = nparts >= 8 ? 0x11111111u : (0x11111111u >> (4 * (8 - nparts)));
            all_present = (x & full) == full && nparts <= 8;
        }
    }
    if (kAccount && (!all_present || throw_after)) {
        for (int o = G >> 1; o > 0; o >>= 1) n_gather += __shfl_xor_sync(gmask, n_gather, o, G);
        if (gl == 0) atomicAdd(a.gather_count, (unsigned long long)n_gather);
    }
    if (!all_present) {  // kmer_index.hpp:224 / :524  return result_t()
        if (PASS == kPassCount && gl == 0) {
            a.counts[q] = 0;
            a.status[q] = KMER_B200_QUERY_OK;
            a.unsorted[q] = 0;
        }
        return;
    }
    if (throw_after) {  // all full parts present, then the rest lookup throws
        if (PASS == kPassCount && gl == 0) {
            a.counts[q] = 0;
            a.status[q] = KMER_B200_QUERY_THROW_INVALID_ARGUMENT;
            a.unsorted[q] = 0;
        }
        return;
    }

    // ---- 4. candidates ---------------------------------------------------------------------------------------
    const Element &E0 = ix.elem[e0];
    uint64_t n_hits = 0;
    bool unsorted = false;
    if (kind == kSubK) {
        // get_position_for_all_kmer_with_prefix (kmer_index.hpp:115-148): the buckets of all hashes in
        // [prefix_hash, prefix_hash + sigma^(k-m)) are one contiguous slab of the sorted position array
        const uint32_t kp = VIEWS ? E0.k_phys : k0;  // a view enumerates the owner's slab: the same positions, the same tail rule
        const uint64_t width = ix.pow_sigma[kp - m];
        const uint64_t lo_key = key_at(qw, 0, m, T.bits, T.sigma) * width;
        const uint64_t slo = lower_bound_key(E0, lo_key);
        const uint64_t shi = lower_bound_key(E0, lo_key + width);
        if (shi - slo > 1) unsorted = element_key_or_text(T, E0, slo) != element_key_or_text(T, E0, shi - 1);
        const bool count_by_range = PASS != kPassWrite && ix.owned == T.n;  // unsharded: every hit is owned
        HAND_OFF_IF_HEAVY(shi - slo)  // same decision in the count and the write pass
        if (count_by_range) n_hits = shi - slo;
        for (uint64_t c0 = slo; c0 < shi && !count_by_range; c0 += G) {
            const uint64_t c = c0 + gl;
            uint32_t p = 0;
            bool ok = false;
            if (c < shi) {
                p = *pos_ptr(E0, c);  // a slab spans buckets, so it may span parts
                ok = (uint64_t)p < ix.owned;
                if (kAccount && ((c & 7) == 0 || c == slo)) ++n_gather;
            }
            const uint32_t b = GBALLOT(ok);
            if (PASS == kPassWrite && ok)
                a.positions[out_base + n_hits + __popc(b & lt_mask)] = p + (uint32_t)ix.global_base;
            n_hits += __popc(b);
        }
        // check_last_kmer (kmer_index.hpp:90-112): starts in the last k-1 positions, where no k-mer starts
        for (uint32_t t0 = 0; t0 < kp - m; t0 += G) {
            const uint32_t t = t0 + gl;
            const uint64_t p = T.n - kp + 1 + t;
            const bool ok = t < kp - m && p < ix.owned && match_span(T, qw, p, 0, m);
            const uint32_t b = GBALLOT(ok);
            if (PASS == kPassWrite && ok)
                a.positions[out_base + n_hits + __popc(b & lt_mask)] = (uint32_t)p + (uint32_t)ix.global_base;
            n_hits += __popc(b);
        }
    } else {
        if (!SINGLE && kind == kBuggySingle && ix.n_elems > 1) {
            // the last full part and the rest are one contiguous stretch of k0 + rest symbols: an element with a
            // larger k (multi-k index) gives a shorter candidate list for it
            const uint32_t last = (P - 1) * k0;
            uint32_t e = e0;
            for (uint32_t i = 0; i < ix.n_elems; ++i) {
                const uint32_t c = ix.elem_by_k_desc[i];
                if (ix.elem[c].k <= k0 + rest) {
                    e = c;
                    break;
                }
            }
            if (ix.elem[e].k > k0) {
                Range alt{0, 0};
                if (gl == 0) {
                    const Element &E = ix.elem[e];
                    alt = bucket_of<VIEWS>(E, key_at(qw, (uint64_t)last, E.k, T.bits, T.sigma));
                    if (kAccount) n_gather += 1 + (E.shift ? 1 : 0);
                }
                alt.lo = GSHFL(alt.lo, 0);
                alt.cnt = GSHFL(alt.cnt, 0);
                // (views: a candidate list is the slab plus the tail starts that are compared directly)
                const uint32_t alt_tail = VIEWS ? ix.elem[e].k_phys - ix.elem[e].k : 0u;
                const uint32_t cur_tail = VIEWS ? ix.elem[seed_e].k_phys - ix.elem[seed_e].k : 0u;
                if (alt.cnt + alt_tail < seed.cnt + cur_tail) {
                    seed = alt;
                    seed_e = e;
                    seed_d = last;
                    if (VIEWS) seed_o = last;
                }
            }
        }
        const Element &Es = ix.elem[seed_e];
        const uint32_t ks = Es.k;
        const uint32_t kf = from_list ? ix.elem[S[0]].k : k0;  // k of part 0 (text stride of the multi-k defect)
        const uint32_t n_spans = kind == kExact ? 0u : (kind == kContig ? 1u : (kind == kBuggySingle ? P : nparts));
        // a view's bucket: slab entries first, then the tail starts (all beyond every slab entry), compared directly
        const uint32_t tail_slots = VIEWS ? Es.k_phys - ks : 0u;
        const uint64_t n_cand = seed.cnt + tail_slots;
        unsorted = VIEWS && Es.width != 1 && seed.cnt > 1;
        bool count_by_range = PASS != kPassWrite && kind == kExact && ix.owned == T.n;
        HAND_OFF_IF_HEAVY(seed.cnt)  // same decision in the count and the write pass
        if (count_by_range) n_hits = seed.cnt;
        if (PASS == kPassWrite && kind == kExact && ix.owned == T.n) {
            // the whole bucket is the result: a plain copy with 8 independent loads in flight per lane
            const uint32_t *src = pos_ptr(Es, seed.lo);
            uint32_t *dst = a.positions + out_base;
            const uint32_t gb = (uint32_t)ix.global_base;
            uint64_t c = gl;
            for (; c + 7 * G < seed.cnt; c += 8 * G) {
                uint32_t v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = src[c + j * G];
#pragma unroll
                for (int j = 0; j < 8; ++j) dst[c + j * G] = v[j] + gb;
            }
            for (; c < seed.cnt; c += G) dst[c] = src[c] + gb;
            count_by_range = true;  // the generic loop below starts behind the slab
            n_hits = seed.cnt;
        }
        // a bucket lies in one part of a peer-positions index; a view's slab (VIEWS) only exists on a whole array
        const uint32_t *cand = pos_ptr(Es, seed.lo);
        for (uint64_t c0 = count_by_range ? seed.cnt : 0; c0 < n_cand; c0 += G) {
            const uint64_t c = c0 + gl;
            uint32_t p = 0;
            bool ok = false;
            if (c < n_cand) {
                uint32_t at;
                if (!VIEWS || c < seed.cnt) {
                    at = gather32(cand + c);
                    ok = true;
                } else {
                    at = (uint32_t)(T.n - Es.k_phys + 1 + (c - seed.cnt));
                    ok = match_span(T, qw, at, seed_o, ks);
                }
                ok = ok && at >= seed_d;
                p = at - seed_d;
                ok = ok && (uint64_t)p < ix.owned;
                if (kAccount && (((seed.lo + c) & 7) == 0 || c == 0)) ++n_gather;
                if (kAccount && ok && kind != kExact) n_gather += 1 + (m * T.bits >> 8);
                // the rest of the plan as text spans (text offset, query offset, length) relative to the match start;
                // one loop for every plan, so the text reads of a warp's lanes are issued together
                for (uint32_t sp = 0; ok && sp < n_spans; ++sp) {
                    uint32_t dt, qo, ln;
                    if (kind == kContig) {
                        dt = ks, qo = ks, ln = m - ks;
                    } else if (SINGLE || kind == kBuggySingle) {
                        // part 0 in place, the middle parts compared against the LAST part (kmer_index.hpp:314),
                        // then the last part and the rest as one stretch
                        const uint32_t last = (P - 1) * k0;
                        dt = sp == 0 ? 0 : (sp + 1 == P ? last : sp * k0);
                        qo = sp == 0 ? 0 : last;
                        ln = sp + 1 == P ? k0 + rest : k0;
                    } else {
                        // part i is read at query offset k_{i-1} and expected at text offset i * k_0
                        // (kmer_index.hpp:526 and :535,544)
                        dt = sp * kf;
                        qo = sp ? ix.elem[S[sp - 1]].k : 0;
                        ln = ix.elem[S[sp]].k;
                    }
                    ok = match_span(T, qw, (uint64_t)p + dt, qo, ln);
                }
            }
            const uint32_t b = GBALLOT(ok);
            if (PASS == kPassWrite && ok)
                a.positions[out_base + n_hits + __popc(b & lt_mask)] = p + (uint32_t)ix.global_base;
            n_hits += __popc(b);
        }
    }
    if (kAccount) {
        if (kind == kSubK && gl == 0) n_gather += 2;  // the two directory lookups of the slab bounds
        for (int o = G >> 1; o > 0; o >>= 1) n_gather += __shfl_xor_sync(gmask, n_gather, o, G);
        if (gl == 0) atomicAdd(a.gather_count, (unsigned long long)n_gather);
    }
    if (PASS == kPassCount && gl == 0) {
        a.counts[q] = n_hits;
        a.status[q] = KMER_B200_QUERY_OK;
        const bool flag = unsorted && n_hits > 1;
        a.unsorted[q] = (flag ? 1 : 0) | (HEAVY ? 2 : 0);
        if (flag) atomicAdd(a.error_flag + 1, 1u);  // number of segments the sort pass has to visit
        if (a.hits != nullptr && n_hits > 0) {
            // the write pass only visits the queries listed here (one atomic per set of lanes arriving together)
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

template <int PASS, int G, bool SINGLE>
__global__ void __launch_bounds__(kSearchThreads, KB_SEARCH_MIN_BLOCKS) search_kernel(const SearchArgs a) {
    constexpr int kGroups = kSearchThreads / G;
    extern __shared__ uint64_t smem_q[];
    const uint64_t q = (uint64_t)blockIdx.x * kGroups + threadIdx.x / G;
    if (q < a.n_queries) search_query<PASS, G, false, SINGLE>(a, q, smem_q);
}

// write pass over the queries the count pass listed as having hits (a.hits[0] = length, a.hits[1..] = query ids):
// with random queries over a large key space that is a small share of the batch, and the lanes of a warp are all busy
template <int G, bool SINGLE>
__global__ void __launch_bounds__(kSearchThreads, KB_SEARCH_MIN_BLOCKS) search_listed_write_kernel(const SearchArgs a) {
    constexpr int kGroups = kSearchThreads / G;
    extern __shared__ uint64_t smem_q[];
    const uint32_t n_listed = a.hits[0];
    for (uint64_t i = (uint64_t)blockIdx.x * kGroups + threadIdx.x / G; i < n_listed; i += (uint64_t)gridDim.x * kGroups) {
        search_query<kPassWrite, G, false, SINGLE>(a, (uint64_t)a.hits[1 + i], smem_q);
        __syncwarp();
    }
}

// second launch of a pass: one warp per query of the heavy list (a.heavy[0] = length, a.heavy[1..] = query ids)
template <int PASS, bool SINGLE>
__global__ void __launch_bounds__(kSearchThreads) search_heavy_kernel(const SearchArgs a) {
    constexpr int kGroups = kSearchThreads / 32;
    extern __shared__ uint64_t smem_q[];
    const uint32_t n_heavy = a.heavy[0];
    for (uint32_t i = blockIdx.x * kGroups + threadIdx.x / 32; i < n_heavy; i += gridDim.x * kGroups) {
        search_query<PASS, 32, true, SINGLE>(a, (uint64_t)a.heavy[1 + i], smem_q);
        __syncwarp();
    }
}

// Shared-positions index: one warp per query (slabs are long), every pass of the unsharded search.
template <int PASS>
__global__ void __launch_bounds__(kSearchThreads) search_views_kernel(const SearchArgs a) {
    constexpr int kGroups = kSearchThreads / 32;
    extern __shared__ uint64_t smem_q[];
    if (PASS == kPassWrite && a.hits != nullptr) {
        const uint32_t n_listed = a.hits[0];
        for (uint64_t i = (uint64_t)blockIdx.x * kGroups + threadIdx.x / 32; i < n_listed; i += (uint64_t)gridDim.x * kGroups) {
            search_query<PASS, 32, false, false, true>(a, (uint64_t)a.hits[1 + i], smem_q);
            __syncwarp();
        }
    } else {
        for (uint64_t q = (uint64_t)blockIdx.x * kGroups + threadIdx.x / 32; q < a.n_queries; q += (uint64_t)gridDim.x * kGroups) {
            search_query<PASS, 32, false, false, true>(a, q, smem_q);
            __syncwarp();
        }
    }
}

template <int PASS>
static void launch_search_views(const SearchArgs &args, cudaStream_t stream) {
    SearchArgs h = args;
    h.group = 32;
    h.q_words = search_q_words(32, args.bits, args.max_len);
    constexpr int kGroups = kSearchThreads / 32;
    const size_t smem = (size_t)kGroups * h.q_words * sizeof(uint64_t);
    const uint64_t blocks = std::min<uint64_t>((args.n_queries + kGroups - 1) / kGroups, (uint64_t)device_sm_count() * 16);
    cudaFuncSetAttribute(search_views_kernel<PASS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    search_views_kernel<PASS><<<(unsigned)blocks, kSearchThreads, smem, stream>>>(h);
}

template <int PASS, int G, bool SINGLE>
static void launch_search_pgs(const SearchArgs &args, cudaStream_t stream) {
    constexpr int kGroups = kSearchThreads / G;
    const uint64_t blocks = (args.n_queries + kGroups - 1) / kGroups;
    const size_t smem = (size_t)kGroups * args.q_words * sizeof(uint64_t);
    cudaFuncSetAttribute(search_kernel<PASS, G, SINGLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (PASS == kPassWrite && args.hits != nullptr) {
        cudaFuncSetAttribute(search_listed_write_kernel<G, SINGLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        search_listed_write_kernel<G, SINGLE>
            <<<(unsigned)std::min<uint64_t>(blocks, (uint64_t)device_sm_count() * 8 * 2), kSearchThreads, smem, stream>>>(args);
    } else {
        search_kernel<PASS, G, SINGLE><<<(unsigned)blocks, kSearchThreads, smem, stream>>>(args);
    }
    if (G < 32 && args.heavy != nullptr && PASS != kPassPresence) {
        // queries with long candidate lists, if any (the list length lives on the device: fixed grid, no host sync)
        SearchArgs h = args;
        h.q_words = search_q_words(32, args.bits, args.max_len);
        const size_t hsmem = (size_t)(kSearchThreads / 32) * h.q_words * sizeof(uint64_t);
        cudaFuncSetAttribute(search_heavy_kernel<PASS, SINGLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem);
        search_heavy_kernel<PASS, SINGLE><<<device_sm_count() * 2, kSearchThreads, hsmem, stream>>>(h);
    }
}

template <int PASS, int G>
static void launch_search_pg(const SearchArgs &args, cudaStream_t stream) {
    if (args.single_k)
        launch_search_pgs<PASS, G, true>(args, stream);
    else
        launch_search_pgs<PASS, G, false>(args, stream);
}

// epilogue of the deferred count pass: the whole-text presence rule (kmer_index.hpp:216-227, :234 -> :119)
__global__ void __launch_bounds__(256) finalize_deferred_kernel(uint64_t *__restrict__ counts, uint8_t *__restrict__ status,
                                                                const uint8_t *__restrict__ defer,
                                                                const uint32_t *__restrict__ present4_global, uint64_t n) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const uint32_t d = defer[q];
    if (!(d & 0x40u)) return;
    const uint32_t parts = d & 0x3Fu;
    uint32_t x = present4_global[q];
    x = (x | (x >> 1) | (x >> 2) | (x >> 3)) & 0x11111111u;
    const uint32_t full = parts >= 8 ? 0x11111111u : (0x11111111u >> (4 * (8 - parts)));
    const bool all_present = parts <= 8 && (x & full) == full;
    if (!all_present) {
        counts[q] = 0;
    } else if (d & 0x80u) {
        counts[q] = 0;
        status[q] = KMER_B200_QUERY_THROW_INVALID_ARGUMENT;
    }
}

void launch_finalize_deferred(uint64_t *d_counts, uint8_t *d_status, const uint8_t *d_defer, const uint32_t *d_present4_global,
                              uint64_t n_queries, cudaStream_t stream) {
    if (n_queries == 0) return;
    finalize_deferred_kernel<<<(unsigned)((n_queries + 255) / 256), 256, 0, stream>>>(d_counts, d_status, d_defer,
                                                                                        d_present4_global, n_queries);
}

uint32_t search_q_words(uint32_t group, uint32_t bits, uint64_t max_len) {
    // rounds of 8 * group symbols, group * bits / 8 words each, plus two zero words
    const uint32_t lpw = 8 / bits;
    const uint32_t cpl = lpw > group ? lpw / group : 1;
    const uint64_t per_round = 8ull * group * cpl;
    const uint64_t rounds = (std::max<uint64_t>(max_len, 1) + per_round - 1) / per_round;
    return (uint32_t)(rounds * (group * cpl / lpw) + 2);
}

bool launch_search_count_lean(const SearchArgs &a, cudaStream_t stream);  // search_lean.cu

void launch_search(const SearchArgs &args, SearchPass pass, cudaStream_t stream) {
    if (args.n_queries == 0) return;
    if (args.views) {
        if (pass == kPassCount) launch_search_views<kPassCount>(args, stream);
        if (pass == kPassCountAccount) launch_search_views<kPassCountAccount>(args, stream);
        if (pass == kPassWrite) launch_search_views<kPassWrite>(args, stream);
        return;  // the sharded passes do not exist for such an index (capi.cu refuses the combination)
    }
    if (pass == kPassCount && launch_search_count_lean(args, stream)) {
        // the lean kernel answered what it covers; the queries it listed (prefix slabs, long candidate lists) go to the
        // general kernel's warp-per-query launch, as after the general count pass
        SearchArgs h = args;
        h.q_words = search_q_words(32, args.bits, args.max_len);
        const size_t hsmem = (size_t)(kSearchThreads / 32) * h.q_words * sizeof(uint64_t);
        if (args.single_k) {
            cudaFuncSetAttribute(search_heavy_kernel<kPassCount, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem);
            search_heavy_kernel<kPassCount, true><<<device_sm_count() * 2, kSearchThreads, hsmem, stream>>>(h);
        }
        return;
    }
    if (args.group == 1) {
        if (pass == kPassCount) launch_search_pg<kPassCount, 1>(args, stream);
        if (pass == kPassCountAccount) launch_search_pg<kPassCountAccount, 1>(args, stream);
        if (pass == kPassCountDeferred) launch_search_pg<kPassCountDeferred, 1>(args, stream);
        if (pass == kPassCountDeferredAccount) launch_search_pg<kPassCountDeferredAccount, 1>(args, stream);
        if (pass == kPassWrite) launch_search_pg<kPassWrite, 1>(args, stream);
        if (pass == kPassPresence) launch_search_pg<kPassPresence, 1>(args, stream);
    } else if (args.group == 2) {
        if (pass == kPassCount) launch_search_pg<kPassCount, 2>(args, stream);
        if (pass == kPassCountAccount) launch_search_pg<kPassCountAccount, 2>(args, stream);
        if (pass == kPassCountDeferred) launch_search_pg<kPassCountDeferred, 2>(args, stream);
        if (pass == kPassCountDeferredAccount) launch_search_pg<kPassCountDeferredAccount, 2>(args, stream);
        if (pass == kPassWrite) launch_search_pg<kPassWrite, 2>(args, stream);
        if (pass == kPassPresence) launch_search_pg<kPassPresence, 2>(args, stream);
    } else if (args.group == 4) {
        if (pass == kPassCount) launch_search_pg<kPassCount, 4>(args, stream);
        if (pass == kPassCountAccount) launch_search_pg<kPassCountAccount, 4>(args, stream);
        if (pass == kPassCountDeferred) launch_search_pg<kPassCountDeferred, 4>(args, stream);
        if (pass == kPassCountDeferredAccount) launch_search_pg<kPassCountDeferredAccount, 4>(args, stream);
        if (pass == kPassWrite) launch_search_pg<kPassWrite, 4>(args, stream);
        if (pass == kPassPresence) launch_search_pg<kPassPresence, 4>(args, stream);
    } else if (args.group == 8) {
        if (pass == kPassCount) launch_search_pg<kPassCount, 8>(args, stream);
        if (pass == kPassCountAccount) launch_search_pg<kPassCountAccount, 8>(args, stream);
        if (pass == kPassCountDeferred) launch_search_pg<kPassCountDeferred, 8>(args, stream);
        if (pass == kPassCountDeferredAccount) launch_search_pg<kPassCountDeferredAccount, 8>(args, stream);
        if (pass == kPassWrite) launch_search_pg<kPassWrite, 8>(args, stream);
        if (pass == kPassPresence) launch_search_pg<kPassPresence, 8>(args, stream);
    } else {
        if (pass == kPassCount) launch_search_pg<kPassCount, 32>(args, stream);
        if (pass == kPassCountAccount) launch_search_pg<kPassCountAccount, 32>(args, stream);
        if (pass == kPassCountDeferred) launch_search_pg<kPassCountDeferred, 32>(args, stream);
        if (pass == kPassCountDeferredAccount) launch_search_pg<kPassCountDeferredAccount, 32>(args, stream);
        if (pass == kPassWrite) launch_search_pg<kPassWrite, 32>(args, stream);
        if (pass == kPassPresence) launch_search_pg<kPassPresence, 32>(args, stream);
    }
}

// ------------------------------------------------------------------------------------------------
// exclusive scan of the per-query counts (u64), in place; counts[Q] receives the total
// ------------------------------------------------------------------------------------------------
constexpr int kScanThreads = 256;
constexpr int kScanPerThread = 16;
constexpr int kScanBlock = kScanThreads * kScanPerThread;  // 4096

__device__ __forceinline__ uint64_t block_exclusive_scan(uint64_t v, uint64_t *total) {
    __shared__ uint64_t warp_sums[kScanThreads / 32];
    __shared__ uint64_t block_total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t run = 0;
        for (int w = 0; w < kScanThreads / 32; ++w) {
            const uint64_t t = warp_sums[w];
            warp_sums[w] = run;
            run += t;
        }
        block_total = run;
    }
    __syncthreads();
    const uint64_t r = incl - v + warp_sums[warp];
    *total = block_total;
    __syncthreads();
    return r;
}

// Each warp owns 512 consecutive counts and reads them as 16 coalesced rounds of 32.
__global__ void __launch_bounds__(kScanThreads) scan_reduce_kernel(const uint64_t *__restrict__ v, uint64_t n,
                                                                   uint64_t *__restrict__ block_sums) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t wbase = (uint64_t)blockIdx.x * kScanBlock + (uint64_t)warp * (32 * kScanPerThread);
    uint64_t s = 0;
#pragma unroll
    for (int r = 0; r < kScanPerThread; ++r) {
        const uint64_t i = wbase + r * 32 + lane;
        if (i < n) s += v[i];
    }
    uint64_t total;
    block_exclusive_scan(s, &total);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kScanThreads) scan_block_sums_kernel(uint64_t *__restrict__ block_sums, uint64_t n_blocks,
                                                                       uint64_t *__restrict__ grand_total) {
    // single CTA: every thread owns a contiguous slice
    const uint64_t per = (n_blocks + kScanThreads - 1) / kScanThreads;
    const uint64_t b0 = (uint64_t)threadIdx.x * per;
    const uint64_t b1 = b0 + per < n_blocks ? b0 + per : n_blocks;
    uint64_t s = 0;
    for (uint64_t b = b0; b < b1; ++b) s += block_sums[b];
    uint64_t total;
    uint64_t run = block_exclusive_scan(s, &total);
    for (uint64_t b = b0; b < b1; ++b) {
        const uint64_t t = block_sums[b];
        block_sums[b] = run;
        run += t;
    }
    if (threadIdx.x == 0) *grand_total = total;
}

__global__ void __launch_bounds__(kScanThreads) scan_apply_kernel(uint64_t *__restrict__ v, uint64_t n,
                                                                  const uint64_t *__restrict__ block_sums) {
    // coalesced rounds -> shared memory -> each lane scans its 16 consecutive values -> back the same way.
    // Row stride 17 keeps the blocked accesses at most 2-way bank conflicted.
    constexpr int kRow = kScanPerThread + 1;
    __shared__ uint64_t tile[kScanThreads / 32][32 * kRow];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t wbase = (uint64_t)blockIdx.x * kScanBlock + (uint64_t)warp * (32 * kScanPerThread);
    uint64_t *mine = tile[warp];
#pragma unroll
    for (int r = 0; r < kScanPerThread; ++r) {
        const int e = r * 32 + lane;  // element of the warp's segment
        const uint64_t i = wbase + e;
        mine[(e / kScanPerThread) * kRow + (e % kScanPerThread)] = i < n ? v[i] : 0;
    }
    __syncwarp();
    uint64_t x[kScanPerThread];
    uint64_t s = 0;
#pragma unroll
    for (int j = 0; j < kScanPerThread; ++j) {
        x[j] = mine[lane * kRow + j];
        s += x[j];
    }
    uint64_t total;
    uint64_t run = block_exclusive_scan(s, &total) + block_sums[blockIdx.x];
#pragma unroll
    for (int j = 0; j < kScanPerThread; ++j) {
        mine[lane * kRow + j] = run;
        run += x[j];
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < kScanPerThread; ++r) {
        const int e = r * 32 + lane;
        const uint64_t i = wbase + e;
        if (i < n) v[i] = mine[(e / kScanPerThread) * kRow + (e % kScanPerThread)];
    }
}

// ------------------------------------------------------------------------------------------------
// gather probe: independent random 8-byte reads (one 32-byte sector each) from a table much larger than L2,
// 8 in flight per thread. Its sectors/s is the denominator of the search roofline ("gather roofline").
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_probe_kernel(const uint64_t *__restrict__ table, uint64_t n_words,
                                                           uint64_t n_gathers, uint64_t *__restrict__ sink) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t acc = 0;
    for (uint64_t g = t * 8; g < n_gathers; g += stride * 8) {
        uint64_t v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            uint64_t x = (g + j) * 0x9E3779B97F4A7C15ull;
            x ^= x >> 29;
            x *= 0xBF58476D1CE4E5B9ull;
            x ^= x >> 32;
            v[j] = table[x % n_words];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) acc += v[j];
    }
    if (acc == 0x1234567887654321ull) *sink = acc;  // keeps the loads alive
}

void launch_gather_probe(const uint64_t *d_table, uint64_t n_words, uint64_t n_gathers, uint64_t *d_sink,
                         cudaStream_t stream) {
    gather_probe_kernel<<<device_sm_count() * 16, 256, 0, stream>>>(d_table, n_words, n_gathers, d_sink);
}

uint64_t offsets_scan_blocks(uint64_t n_queries) { return (n_queries + kScanBlock - 1) / kScanBlock; }

void launch_offsets_scan(uint64_t *d_counts, uint64_t n_queries, uint64_t *d_block_sums, cudaStream_t stream) {
    const uint64_t blocks = offsets_scan_blocks(n_queries);
    if (n_queries == 0) {
        cudaMemsetAsync(d_counts, 0, sizeof(uint64_t), stream);
        return;
    }
    scan_reduce_kernel<<<(unsigned)blocks, kScanThreads, 0, stream>>>(d_counts, n_queries, d_block_sums);
    scan_block_sums_kernel<<<1, kScanThreads, 0, stream>>>(d_block_sums, blocks, d_counts + n_queries);
    scan_apply_kernel<<<(unsigned)blocks, kScanThreads, 0, stream>>>(d_counts, n_queries, d_block_sums);
}

// ------------------------------------------------------------------------------------------------
// segment sort: ascending sort of each flagged query's positions (sub-k results spanning several
// buckets; the reference's std::sort in to_vector, kmer_index_result.hpp:257). One CTA per query.
// Segments up to kSortTile elements are sorted by a bitonic network in shared memory; longer ones by
// an in-CTA stable LSD radix sort ping-ponging between `positions` and `tmp`.
// ------------------------------------------------------------------------------------------------
struct SegSortSmem {
    RankSmem rank;
    uint32_t base[kRadix];
    uint32_t vals[kSortTile];
};

__global__ void __launch_bounds__(kSortThreads, 1)
    segment_sort_kernel(uint32_t *__restrict__ positions, uint32_t *__restrict__ tmp, const uint64_t *__restrict__ offsets,
                        const uint8_t *__restrict__ unsorted, uint64_t n_queries, uint32_t key_bits) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SegSortSmem &sm = *reinterpret_cast<SegSortSmem *>(smem_raw);
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    for (uint64_t q = blockIdx.x; q < n_queries; q += gridDim.x) {
        if (!(unsorted[q] & 1)) continue;
        const uint64_t seg0 = offsets[q];
        const uint64_t len = offsets[q + 1] - seg0;
        if (len < 2) continue;
        if (len <= (uint64_t)kSortTile) {
            uint32_t np2 = 1;
            while (np2 < len) np2 <<= 1;
            for (uint32_t i = tid; i < np2; i += kSortThreads) sm.vals[i] = i < len ? positions[seg0 + i] : 0xFFFFFFFFu;
            __syncthreads();
            for (uint32_t size = 2; size <= np2; size <<= 1) {
                for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                    for (uint32_t i = tid; i < (np2 >> 1); i += kSortThreads) {
                        const uint32_t lo = 2 * i - (i & (stride - 1));
                        const uint32_t hi = lo + stride;
                        const bool up = (lo & size) == 0;
                        const uint32_t x = sm.vals[lo], y = sm.vals[hi];
                        if ((x > y) == up) {
                            sm.vals[lo] = y;
                            sm.vals[hi] = x;
                        }
                    }
                    __syncthreads();
                }
            }
            for (uint32_t i = tid; i < len; i += kSortThreads) positions[seg0 + i] = sm.vals[i];
            __syncthreads();
            continue;
        }
        // long segment: LSD radix, 8 bits per pass
        uint32_t *src = positions + seg0, *dst = tmp + seg0;
        const uint32_t n_pass = (key_bits + 7) / 8;
        for (uint32_t pass = 0; pass < n_pass; ++pass) {
            const uint32_t shift = pass * 8;
            if (tid < kRadix) sm.base[tid] = 0;
            __syncthreads();
            for (uint64_t i = tid; i < len; i += kSortThreads) atomicAdd(&sm.base[(src[i] >> shift) & 0xFF], 1u);
            __syncthreads();
            if (tid < kRadix) {  // exclusive scan over digits -> running destination of each digit
                const uint32_t c = sm.base[tid];
                uint32_t incl = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                    if (lane >= o) incl += v;
                }
                if (lane == 31) sm.rank.warp_sums[warp] = incl;
                sm.rank.count[tid] = incl - c;
            }
            __syncthreads();
            if (tid < kRadix) {
                uint32_t b = sm.rank.count[tid];
                for (int w = 0; w < warp; ++w) b += sm.rank.warp_sums[w];
                sm.base[tid] = b;
            }
            __syncthreads();
            for (uint64_t t0 = 0; t0 < len; t0 += kSortTile) {
                const uint32_t count = (uint32_t)min((uint64_t)kSortTile, len - t0);
                uint32_t val[kSortItems], local_pos2[kSortItems / 2];
#pragma unroll
                for (int r = 0; r < kSortItems; ++r) {
                    const uint32_t e = (uint32_t)((warp * kSortItems + r) * 32 + lane);
                    val[r] = e < count ? src[t0 + e] : 0u;
                }
                tile_rank<8, false, uint32_t>(val, count, shift, 0xFFu, local_pos2, sm.rank);
#pragma unroll
                for (int r = 0; r < kSortItems; ++r) {
                    const uint32_t e = (uint32_t)((warp * kSortItems + r) * 32 + lane);
                    const uint32_t d = (val[r] >> shift) & 0xFF;
                    if (e < count) dst[sm.base[d] + (((local_pos2[r >> 1] >> (16 * (r & 1))) & 0xFFFFu) - sm.rank.excl[d])] = val[r];
                }
                __syncthreads();
                if (tid < kRadix) sm.base[tid] += sm.rank.count[tid];
                __syncthreads();
            }
            uint32_t *t = src;
            src = dst;
            dst = t;
        }
        if (src != positions + seg0)
            for (uint64_t i = tid; i < len; i += kSortThreads) positions[seg0 + i] = src[i];
        __syncthreads();
    }
}

void launch_segment_sort(uint32_t *d_positions, uint32_t *d_tmp, const uint64_t *d_offsets, const uint8_t *d_unsorted,
                         uint64_t n_queries, uint32_t key_bits, cudaStream_t stream) {
    if (n_queries == 0) return;
    cudaFuncSetAttribute(segment_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SegSortSmem));
    const uint64_t blocks = n_queries < (uint64_t)device_sm_count() * 64 ? n_queries : (uint64_t)device_sm_count() * 64;
    segment_sort_kernel<<<(unsigned)blocks, kSortThreads, sizeof(SegSortSmem), stream>>>(d_positions, d_tmp, d_offsets,
                                                                                        d_unsorted, n_queries, key_bits);
}

}  // namespace kb
