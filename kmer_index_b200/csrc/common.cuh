// Shared device-side definitions for libkmer_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/kmer_b200.h"

namespace kb {

constexpr int kMaxElements = 32;
constexpr int kMaxPosParts = 8;  // Element::pos_part
constexpr uint32_t kQuerySizeRange = 10000;  // kmer_index.hpp:401

// ---------------------------------------------------------------------------------------------
// Packed text. Symbol i occupies `bits` bits (2, 4 or 8), MSB-first inside 64-bit words, so that a
// window of consecutive symbols read as one big-endian bit field IS the reference's positional hash
// for power-of-two alphabets (kmer_index.hpp:56-73: the first symbol carries sigma^(k-1)).
// The word array carries two zero words of padding so a window read never leaves the allocation.
// ---------------------------------------------------------------------------------------------
struct PackedText {
    const uint64_t *words;
    uint64_t n;     // symbols
    uint32_t bits;  // per symbol
    uint32_t sigma;
};

// 64 bits starting at symbol `sym` (left-aligned: the first symbol sits in the top `bits` bits).
template <typename WordPtr>
__device__ __forceinline__ uint64_t window64(WordPtr words, uint64_t sym, uint32_t bits) {
    const uint64_t bit = sym * bits;
    const uint64_t w = bit >> 6;
    const uint32_t sh = (uint32_t)(bit & 63);
    const uint64_t hi = words[w];
    const uint64_t lo = words[w + 1];
    return sh ? ((hi << sh) | (lo >> (64 - sh))) : hi;
}

// Data-dependent reads of the search (directory, buckets, text windows). On sm_100a a default load that misses L2
// costs a 128-byte DRAM fetch; the L2::64B qualifier halves that (profiles/tools/gather_variants.cu: 127 -> 64
// bytes of DRAM traffic per random 8-byte read). The index is immutable while a search runs: non-coherent path.
__device__ __forceinline__ uint32_t gather32(const uint32_t *p) {
    uint32_t v;
    asm("ld.global.nc.L2::64B.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint64_t gather64(const uint64_t *p) {
    uint64_t v;
    asm("ld.global.nc.L2::64B.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}

// window64 over the packed text in global memory, read with gather loads
__device__ __forceinline__ uint64_t text_window64(const uint64_t *words, uint64_t sym, uint32_t bits) {
    const uint64_t bit = sym * bits;
    const uint64_t w = bit >> 6;
    const uint32_t sh = (uint32_t)(bit & 63);
    const uint64_t hi = gather64(words + w);
    const uint64_t lo = gather64(words + w + 1);
    return sh ? ((hi << sh) | (lo >> (64 - sh))) : hi;
}

// T[tpos, tpos+len) == q[qpos, qpos+len), false if the text span leaves the text (qw: the packed query)
__device__ __forceinline__ bool match_span(const PackedText &T, const uint64_t *qw, uint64_t tpos, uint32_t qpos,
                                           uint32_t len) {
    if (tpos + len > T.n) return false;
    const uint32_t spw = 64 / T.bits;
    while (len) {
        const uint32_t c = len < spw ? len : spw;
        const uint64_t a = text_window64(T.words, tpos, T.bits);
        const uint64_t b = window64(qw, (uint64_t)qpos, T.bits);
        if ((a ^ b) >> (64 - c * T.bits)) return false;
        tpos += c;
        qpos += c;
        len -= c;
    }
    return true;
}

// Hamming distance of T[tpos, tpos+len) and q[qpos, qpos+len) (the caller keeps the span inside the text), counted one
// 64-bit window at a time: XOR the windows, OR-fold every b-bit field onto its lowest bit, keep those bits, popcount.
// Returns early with a count above `limit` as soon as the count exceeds it.
__device__ __forceinline__ uint32_t mismatches_span(const PackedText &T, const uint64_t *qw, uint64_t tpos, uint32_t qpos,
                                                    uint32_t len, uint32_t limit) {
    const uint32_t spw = 64 / T.bits;
    const uint64_t low = T.bits == 2 ? 0x5555555555555555ull : (T.bits == 4 ? 0x1111111111111111ull : 0x0101010101010101ull);
    uint32_t d = 0;
    while (len) {
        const uint32_t c = len < spw ? len : spw;
        uint64_t x = text_window64(T.words, tpos, T.bits) ^ window64(qw, (uint64_t)qpos, T.bits);
        x |= x >> 1;
        if (T.bits >= 4) x |= x >> 2;
        if (T.bits == 8) x |= x >> 4;
        x &= low;
        if (c < spw) x &= ~0ull << (64 - c * T.bits);  // the fields of the c symbols at the top
        d += (uint32_t)__popcll(x);
        if (d > limit) return d;
        tpos += c;
        qpos += c;
        len -= c;
    }
    return d;
}

// The k-mer hash of the k symbols at the top of window `w` (kmer_index.hpp:56-73).
// sigma == 4: the 2k-bit field itself. Otherwise Horner over the k symbols (k * bits <= 64).
__device__ __forceinline__ uint64_t key_from_window(uint64_t w, uint32_t k, uint32_t bits, uint32_t sigma) {
    if (sigma == (1u << bits)) return w >> (64 - k * bits);
    uint64_t h = 0;
    const uint64_t mask = (1ull << bits) - 1;
#pragma unroll 1
    for (uint32_t i = 0; i < k; ++i) {
        h = h * sigma + ((w >> (64 - bits * (i + 1))) & mask);
    }
    return h;
}

// Hash of the k symbols starting at symbol `sym`, for any legal k (kmer_index.hpp:42-43). k * bits can exceed one
// window only for alphabets that are not a power of two (aa27 k >= 9, dna5 k >= 17; sigma^k < 2^64 keeps k * bits
// < 64 otherwise): the Horner walk then continues into a second window (k * bits <= 128 always).
template <typename WordPtr>
__device__ __forceinline__ uint64_t key_at(WordPtr words, uint64_t sym, uint32_t k, uint32_t bits, uint32_t sigma) {
    const uint64_t w0 = window64(words, sym, bits);
    const uint32_t spw = 64 / bits;
    if (k <= spw) return key_from_window(w0, k, bits, sigma);
    const uint64_t w1 = window64(words, sym + spw, bits);
    const uint64_t mask = (1ull << bits) - 1;
    uint64_t h = 0;
#pragma unroll 1
    for (uint32_t i = 0; i < spw; ++i) h = h * sigma + ((w0 >> (64 - bits * (i + 1))) & mask);
#pragma unroll 1
    for (uint32_t i = 0; i < k - spw; ++i) h = h * sigma + ((w1 >> (64 - bits * (i + 1))) & mask);
    return h;
}

// ---------------------------------------------------------------------------------------------
// One index element (one k): the CSR form of the reference's
// robin_hood::unordered_map<hash, std::vector<position>> (kmer_index.hpp:52).
//   pos[n_kmers]   all k-mer start positions, stably sorted by hash (bucket = run of equal hashes,
//                  ascending positions inside, as push_back in text order yields, kmer_index.hpp:165)
//   dir[entries]   dir[j] = number of k-mers with (hash >> shift) < j      (entries = (max_hash >> shift) + 2)
//   keys[n_kmers]  the sorted hashes, kept only when the directory is not dense (shift > 0: lookups finish with a
//                  binary search in them); null for a dense directory -- a hash is then recomputed from the text at
//                  pos[i] where one is needed. 32-bit while sigma^k <= 2^32, 64-bit otherwise.
// ---------------------------------------------------------------------------------------------
struct Element {
    uint32_t k;
    uint32_t shift;
    uint64_t n_kmers;
    uint64_t dir_entries;
    uint64_t key_space;  // sigma^k
    const uint32_t *dir;
    const void *keys;
    const uint32_t *pos;
    uint32_t key_bytes;  // 4 or 8
    uint32_t k_phys;     // == k, except for a VIEW (below)
    uint64_t key_lo, key_hi;  // the element indexes the k-mers with hash in [key_lo, key_hi): a key-range part of a
                              // multi-GPU build, else [0, 2^64 - 1]; dir and keys are relative to key_lo
    // Shared-positions multi-k index (SURVEY.md 8f.2, thesis outlook 04_outlook_and_conclusion.tex:25-45): only the
    // element with the largest k (k_phys) owns arrays; a smaller k is a VIEW of them -- dir / keys / pos / shift /
    // n_kmers / key_space are the owner's, and the bucket of k-mer hash h is the slab of the sigma^(k_phys - k)
    // consecutive k_phys-mer hashes that start with it: [h * width, (h + 1) * width). Inside a slab the positions are
    // ordered by the following k_phys - k symbols, not by position, and the last k_phys - k k-mer starts of the text
    // (where no k_phys-mer starts) are not in it: the search compares those "tail" starts directly and sorts what it
    // reports. width == 1 for an ordinary element.
    uint64_t width;
    // Peer-positions multi-GPU index (n_pos_parts > 0, pos == null): the position array stays cut into the key-range
    // parts the GPUs built -- part r holds the CSR entries [part_first[r], part_first[r + 1]) in pos_part[r], which is
    // this GPU's memory for one r and another GPU's memory, mapped over NVLink, for the others. Part boundaries are
    // bucket boundaries, so a bucket lies in one part. The directory is whole on every GPU.
    uint32_t n_pos_parts;
    uint32_t part_first[kMaxPosParts + 1];
    const uint32_t *pos_part[kMaxPosParts];
};

// address of CSR entry i of element E
__device__ __forceinline__ const uint32_t *pos_ptr(const Element &E, uint64_t i) {
    if (E.n_pos_parts == 0) return E.pos + i;
    uint32_t r = 0;
#pragma unroll
    for (uint32_t j = 1; j < (uint32_t)kMaxPosParts; ++j) r += (j < E.n_pos_parts && i >= (uint64_t)E.part_first[j]) ? 1u : 0u;
    return E.pos_part[r] + (i - E.part_first[r]);
}

__device__ __forceinline__ uint64_t element_key(const Element &E, uint64_t i) {
    return E.key_bytes == 8 ? gather64(static_cast<const uint64_t *>(E.keys) + i)
                            : (uint64_t)gather32(static_cast<const uint32_t *>(E.keys) + i);
}
// same, for elements that may not hold their hashes (dense directory): recomputed from the text at pos[i]
__device__ __forceinline__ uint64_t element_key_or_text(const PackedText &T, const Element &E, uint64_t i) {
    if (E.keys != nullptr) return element_key(E, i);
    return key_at(T.words, (uint64_t)gather32(pos_ptr(E, i)), E.k_phys, T.bits, T.sigma);
}

// ---- directory lookups (the reference's at(hash), kmer_index.hpp:76-84) ------------------------------------------------
struct Range {
    uint64_t lo;
    uint64_t cnt;
};

// index of the first sorted k-mer of element E whose hash is >= key (key may equal key_space)
__device__ __forceinline__ uint64_t lower_bound_key(const Element &E, uint64_t key) {
    if (key >= E.key_space || key >= E.key_hi) return E.n_kmers;
    if (key <= E.key_lo) return 0;
    key -= E.key_lo;
    const uint64_t t = key >> E.shift;
    uint64_t lo = gather32(E.dir + t);
    if (E.shift == 0) return lo;
    uint64_t hi = gather32(E.dir + t + 1);
    while (lo < hi) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        if (element_key(E, mid) < key)
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo;
}

// the bucket of `key`: the reference's at(hash) (kmer_index.hpp:76-84)
template <bool VIEWS = false>
__device__ __forceinline__ Range bucket_of(const Element &E, uint64_t key) {
    if (VIEWS && E.width != 1) {  // a view: the slab of the owner's hashes that start with `key` (tail starts: see Element)
        const uint64_t lo = lower_bound_key(E, key * E.width);
        return Range{lo, lower_bound_key(E, (key + 1) * E.width) - lo};
    }
    if (key < E.key_lo || key >= E.key_hi) return Range{0, 0};  // another part's hash
    key -= E.key_lo;
    const uint64_t t = key >> E.shift;
    uint64_t lo = gather32(E.dir + t);
    uint64_t hi = gather32(E.dir + t + 1);
    if (E.shift != 0) {
        uint64_t a = lo, b = hi;
        while (a < b) {
            const uint64_t mid = a + ((b - a) >> 1);
            if (element_key(E, mid) < key)
                a = mid + 1;
            else
                b = mid;
        }
        lo = a;
        b = hi;
        while (a < b) {
            const uint64_t mid = a + ((b - a) >> 1);
            if (element_key(E, mid) <= key)
                a = mid + 1;
            else
                b = mid;
        }
        hi = a;
    }
    return Range{lo, hi - lo};
}

struct SchemeTables {
    // row m of the reference's _optimal_nk_sum / _use_multi_search_scheme (kmer_index.hpp:404-405),
    // with ks replaced by element indices
    const uint32_t *sum_off;   // [kQuerySizeRange + 1]
    const uint8_t *sum_elem;   // flattened lists
    const uint8_t *use_multi;  // [kQuerySizeRange]
};

struct DeviceIndex {
    PackedText text;
    uint64_t owned;        // match starts p are reported only for p < owned (sharding); == n unsharded
    uint64_t global_base;  // added to every reported position (shard_begin)
    uint32_t n_elems;
    uint32_t sharded;
    Element elem[kMaxElements];
    SchemeTables scheme;
    uint64_t pow_sigma[64];  // sigma^e for e < 64 (saturating at 2^63)
    uint8_t elem_by_k_desc[kMaxElements];  // element indices ordered by k descending (_all_ks, :410)
    // Auxiliary elements (slots n_elems..): an index with k' = m built on demand for a query length m that the
    // plan answers by prefix enumeration (m < k). The bucket of the whole query in the k' = m index IS the
    // sorted union of the sigma^(k-m) buckets the reference enumerates (kmer_index.hpp:138-144) plus the
    // end-of-text positions of check_last_kmer (:90-112), so the result is identical and needs no sort.
    uint8_t aux_for_len[64];  // element slot for query length m < 64, 0xFF = none
    // key-range multi-GPU search: per element, a bitmap over the WHOLE key space (bit h = hash h occurs in the text),
    // or null. With it a part answers "does this part of the query occur anywhere" for hashes other parts own.
    const uint64_t *presence[kMaxElements];
    // Collection index (kmer_b200_attach_records), else null / zero: bit s of `boundary` is set for every record start
    // 0 < s < n, so a window [p, p+m) lies inside one record exactly when no bit of [p+1, p+m) is set. Per query length
    // m = 1..8 (the "every window" answer of m <= e): n_win[m] = in-record windows, first_win[m] = the lowest one.
    const uint64_t *boundary;
    uint64_t n_win[9];
    uint64_t first_win[9];
};

// no record of a collection index starts inside (p, p+m): ceil(m / 64) + 1 words at most, read like the text
__device__ __forceinline__ bool window_in_record(const uint64_t *boundary, uint64_t p, uint32_t m) {
    if (m <= 1) return true;
    const uint64_t a = p + 1, b = p + m - 1;  // the bits [a, b]
    uint64_t w = a >> 6;
    const uint64_t w_last = b >> 6;
    uint64_t x = gather64(boundary + w) & (~0ull << (a & 63));
    while (w < w_last) {
        if (x) return false;
        x = gather64(boundary + ++w);
    }
    const uint32_t hb = (uint32_t)(b & 63);
    if (hb != 63) x &= (2ull << hb) - 1;
    return x == 0;
}

}  // namespace kb
