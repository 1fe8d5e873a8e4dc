// Device-side packing of queries: 1 byte per rank -> the text's b-bit MSB-first words (used by the search kernels, which
// pack into shared memory, and by the query router of the key-range multi-GPU search).
#pragma once

#include "common.cuh"

namespace kb {

// ---- query packing helpers ----------------------------------------------------------------------------
// 8 ranks held as the bytes of v (byte j = symbol j) -> 8*bits bits, symbol 0 in the most significant field
__device__ __forceinline__ uint64_t pack8(uint64_t v, uint32_t bits) {
    const uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
    if (bits == 2) {
        // four 2-bit fields at bits 0, 8, 16, 24 -> one byte, field 0 on top: the multiplier 2^30 + 2^20 + 2^10 + 1
        // brings field i to bit 30 - 2i; every cross term lands below bit 24 on a position of its own (no carries)
        // or above bit 31 (dropped by the 32-bit product)
        return (uint64_t)((((lo * 0x40100401u) >> 24) << 8) | ((hi * 0x40100401u) >> 24));
    }
    if (bits == 4) {
        uint32_t a = __byte_perm(lo, 0, 0x0123), b = __byte_perm(hi, 0, 0x0123);  // field 0 to the top byte
        a = (a | (a >> 4)) & 0x00FF00FFu;
        b = (b | (b >> 4)) & 0x00FF00FFu;
        a = (a | (a >> 8)) & 0xFFFFu;
        b = (b | (b >> 8)) & 0xFFFFu;
        return (uint64_t)((a << 16) | b);
    }
    return ((uint64_t)__byte_perm(lo, 0, 0x0123) << 32) | __byte_perm(hi, 0, 0x0123);  // byte reversal
}

// 8 query bytes starting at p (unaligned), bytes >= n_valid zeroed. `safe` = [p, p + 16) lies inside the buffer.
__device__ __forceinline__ uint64_t load8(const uint8_t *p, uint32_t n_valid, bool safe) {
    uint64_t v;
    if (safe) {
        const uint64_t *a = reinterpret_cast<const uint64_t *>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)7);
        const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 7) * 8;
        const uint64_t lo = a[0];
        v = lo;
        if (sh) v = (lo >> sh) | (a[1] << (64 - sh));
    } else {
        v = 0;
        for (uint32_t j = 0; j < 8 && j < n_valid; ++j) v |= (uint64_t)p[j] << (8 * j);
    }
    if (n_valid < 8) v &= (1ull << (8 * n_valid)) - 1;
    return v;
}

// sigma > 128: the per-byte range check (the bit-7 trick below needs sigma <= 128). Rare enough to stay out of line.
static __device__ __noinline__ bool any_rank_out_of_range(const uint8_t *qr, uint32_t m, uint32_t sigma) {
    bool bad = false;
    for (uint32_t i = 0; i < m; ++i) bad |= qr[i] >= sigma;
    return bad;
}

// G = 1: one lane packs its whole query into qw[] (+ two zero words). Returns true when a rank is >= sigma.
// The bytes of one packed word (64 / BITS symbols) are fetched as 8 / BITS + 1 aligned 8-byte words -- each
// once, all in flight together -- and funnel-shifted by the query's misalignment, which is the same for every
// word of the query because a packed word covers a multiple of 8 bytes.
template <int BITS>
__device__ __forceinline__ bool pack_query_lane(const uint8_t *__restrict__ q_ranks, uint64_t off0, uint32_t m,
                                                uint64_t q_total, uint32_t sigma, uint64_t *qw) {
    constexpr int LPW = 8 / BITS;         // 8-symbol chunks per packed word
    constexpr uint32_t SPW = 64 / BITS;   // symbols (= query bytes) per packed word
    const uint8_t *qr = q_ranks + off0;
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(qr) & 7);
    const uint32_t sh = (mis & 3) * 8;
    const bool odd = mis >= 4;
    const uint64_t guard = (0x80u - (sigma > 128 ? 128u : sigma)) * 0x0101010101010101ull;
    uint64_t inval = 0;  // bit 7 of a byte ends up set <=> that rank is >= sigma (sigma <= 128)
    const uint32_t n_words = (m + SPW - 1) / SPW;
    for (uint32_t w = 0; w < n_words; ++w) {
        const uint32_t s0 = w * SPW;
        const uint32_t n_sym = min(SPW, m - s0);
        uint64_t v[LPW];
        if (off0 + s0 >= 8 && off0 + s0 + SPW + 8 <= q_total) {  // the LPW + 1 aligned words lie inside the batch
            const uint64_t *ap = reinterpret_cast<const uint64_t *>(qr + s0 - mis);
            uint32_t r[2 * LPW + 2];
#pragma unroll
            for (int i = 0; i <= LPW; ++i) {
                const uint64_t x = ap[i];
                r[2 * i] = (uint32_t)x;
                r[2 * i + 1] = (uint32_t)(x >> 32);
            }
#pragma unroll
            for (int c = 0; c < LPW; ++c) {
                const uint32_t A = odd ? r[2 * c + 1] : r[2 * c];
                const uint32_t B = odd ? r[2 * c + 2] : r[2 * c + 1];
                const uint32_t C = odd ? r[2 * c + 3] : r[2 * c + 2];
                v[c] = ((uint64_t)__funnelshift_r(B, C, sh) << 32) | __funnelshift_r(A, B, sh);
            }
        } else {  // the first and the last few queries of a batch: byte by byte
#pragma unroll
            for (int c = 0; c < LPW; ++c) v[c] = (uint32_t)(8 * c) < n_sym ? load8(qr + s0 + 8 * c, n_sym - 8 * c, false) : 0ull;
        }
        if (n_sym < SPW) {  // the query ends inside this word: drop the bytes behind it
#pragma unroll
            for (int c = 0; c < LPW; ++c) {
                const uint32_t nv = n_sym > (uint32_t)(8 * c) ? n_sym - 8 * c : 0u;
                if (nv < 8) v[c] &= (1ull << (8 * nv)) - 1;
            }
        }
        uint64_t acc = 0;
#pragma unroll
        for (int c = 0; c < LPW; ++c) {
            inval |= (v[c] + guard) | v[c];
            acc |= pack8(v[c], BITS) << (64 - 8 * BITS * (c + 1));
        }
        qw[w] = acc;
    }
    qw[n_words] = 0;
    qw[n_words + 1] = 0;
    if (sigma > 128) return any_rank_out_of_range(qr, m, sigma);
    return (inval & 0x8080808080808080ull) != 0;
}

// One group of G lanes (lane gl of the group, warp mask gmask) packs the m ranks at q_ranks[off0..] into qw[] (b bits per
// symbol, MSB-first, + two zero words) and sets bit 0 of *error_flag when a rank is >= sigma. q_total = symbols in
// q_ranks (bounds the 16-byte reads). A chunk is 8 symbols (one 8-byte load); `lpw` chunks make one 64-bit word. Each
// lane takes `cpl` consecutive chunks per round so that a round always covers whole words; lanes sharing a word combine
// their parts with xor-shuffles. The group is converged on return.
template <int G>
__device__ __forceinline__ void pack_query_group(const uint8_t *q_ranks, uint64_t off0, uint32_t m, uint64_t q_total,
                                                 const PackedText &T, uint32_t gl, uint32_t gmask, uint32_t *error_flag,
                                                 uint64_t *qw) {
    const uint8_t *qr = q_ranks + off0;
    const uint32_t lpw = 8 / T.bits;                          // chunks per word: 4, 2, 1
    const uint32_t cpl = lpw > (uint32_t)G ? lpw / G : 1;     // chunks per lane and round
    const uint32_t share = lpw / cpl;                         // lanes sharing one word
    const uint32_t wpr = (uint32_t)G * cpl / lpw;             // words per round
    const uint64_t guard = (0x80u - (T.sigma > 128 ? 128u : T.sigma)) * 0x0101010101010101ull;
    bool bad = false;
    uint32_t round = 0;
    if (G == 1) {
        if (T.bits == 2) bad = pack_query_lane<2>(q_ranks, off0, m, q_total, T.sigma, qw);
        else if (T.bits == 4) bad = pack_query_lane<4>(q_ranks, off0, m, q_total, T.sigma, qw);
        else bad = pack_query_lane<8>(q_ranks, off0, m, q_total, T.sigma, qw);
    } else
    for (uint32_t base = 0; base < m; base += 8 * G * cpl, ++round) {
        uint64_t w = 0;
        for (uint32_t c = 0; c < cpl; ++c) {
            const uint32_t chunk = gl * cpl + c;              // chunk index inside the round
            const uint32_t s0 = base + 8 * chunk;
            uint64_t v = 0;
            if (s0 < m) {
                v = load8(qr + s0, m - s0, off0 + s0 + 16 <= q_total);
                if (T.sigma <= 128) {
                    bad |= (((v + guard) | v) & 0x8080808080808080ull) != 0;
                } else {
                    for (uint32_t j = 0; j < 8; ++j) bad |= ((v >> (8 * j)) & 0xFF) >= T.sigma;
                }
            }
            w |= pack8(v, T.bits) << (64 - 8 * T.bits * ((chunk % lpw) + 1));
        }
        for (uint32_t o = 1; o < share; o <<= 1) w |= __shfl_xor_sync(gmask, w, o, G);
        if (gl % share == 0) qw[round * wpr + gl / share] = w;
    }
    if (G > 1 && gl == 0) {
        qw[round * wpr] = 0;
        qw[round * wpr + 1] = 0;
    }
    if ((G == 1 ? bad : __any_sync(gmask, bad)) && gl == 0) atomicOr(error_flag, 1u);
    if (G > 1) __syncwarp(gmask);
}

}  // namespace kb
