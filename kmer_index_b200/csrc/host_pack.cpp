// See host_pack.h. Plain C++ (no CUDA): compiled by the host compiler through nvcc.
#include "host_pack.h"

#include <immintrin.h>

#include <algorithm>
#include <condition_variable>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

namespace kb {

struct HostPool::Impl {
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    std::function<void(unsigned)> fn;
    unsigned n_tasks = 0, next = 0, running = 0;
    uint64_t generation = 0;
    bool stop = false;

    void loop() {
        uint64_t seen = 0;
        std::unique_lock<std::mutex> lock(mu);
        for (;;) {
            cv_work.wait(lock, [&] { return stop || (generation != seen && next < n_tasks); });
            if (stop) return;
            while (next < n_tasks) {
                const unsigned i = next++;
                ++running;
                lock.unlock();
                fn(i);
                lock.lock();
                --running;
            }
            seen = generation;
            if (running == 0) cv_done.notify_all();
        }
    }
};

HostPool::HostPool() : impl_(new Impl) {
    unsigned n = std::thread::hardware_concurrency();
    n = std::max(1u, std::min(n, 32u));
    for (unsigned t = 0; t < n; ++t) impl_->workers.emplace_back([this] { impl_->loop(); });
}

HostPool::~HostPool() {
    {
        std::lock_guard<std::mutex> lock(impl_->mu);
        impl_->stop = true;
    }
    impl_->cv_work.notify_all();
    for (auto &w : impl_->workers) w.join();
    delete impl_;
}

HostPool &HostPool::instance() {
    static HostPool pool;
    return pool;
}

unsigned HostPool::threads() const { return (unsigned)impl_->workers.size(); }

void HostPool::submit(unsigned n_tasks, std::function<void(unsigned)> fn) {
    std::unique_lock<std::mutex> lock(impl_->mu);
    impl_->cv_done.wait(lock, [&] { return impl_->next >= impl_->n_tasks && impl_->running == 0; });
    impl_->fn = std::move(fn);
    impl_->n_tasks = n_tasks;
    impl_->next = 0;
    ++impl_->generation;
    lock.unlock();
    impl_->cv_work.notify_all();
}

void HostPool::wait() {
    std::unique_lock<std::mutex> lock(impl_->mu);
    impl_->cv_done.wait(lock, [&] { return impl_->next >= impl_->n_tasks && impl_->running == 0; });
}

uint64_t query_lengths_host(const uint64_t *q_offsets, uint64_t q_begin, uint64_t q_end, uint16_t *lens, unsigned part,
                            unsigned n_parts) {
    const uint64_t n = q_end - q_begin;
    const uint64_t lo = q_begin + n * part / n_parts, hi = q_begin + n * (part + 1) / n_parts;
    uint64_t mx = 0;
    for (uint64_t i = lo; i < hi; ++i) {
        const uint64_t m = q_offsets[i + 1] - q_offsets[i];
        lens[i - q_begin] = (uint16_t)m;
        mx = std::max(mx, m);
    }
    return mx;
}

namespace {

// 8 ranks (byte j = symbol j) -> 8 * bits bits, symbol 0 on top. This file is compiled for x86-64-v3 (BMI2: one PEXT
// per 8 symbols); the shift-and-mask form is the portable fallback.
template <int BITS>
inline uint64_t pack8(uint64_t v) {
#if defined(__BMI2__)
    constexpr uint64_t mask = BITS == 2 ? 0x0303030303030303ull : BITS == 4 ? 0x0F0F0F0F0F0F0F0Full : ~0ull;
    return _pext_u64(__builtin_bswap64(v), mask);
#else
    uint64_t r = 0;
    for (int j = 0; j < 8; ++j) r |= ((v >> (8 * j)) & ((1ull << BITS) - 1)) << (BITS * (7 - j));
    return r;
#endif
}

// ---- streaming pack: a contiguous run of ranks -> words, query boundaries ignored ---------------------------------
#if defined(__AVX2__)
// 32 four-bit ranks -> two 64-bit words (16 symbols each)
static inline void pack32x4(__m256i v, uint64_t &w0, uint64_t &w1) {
    const __m256i x = _mm256_maddubs_epi16(v, _mm256_set1_epi16(0x0110));  // 16 a + b in every 16-bit lane
    const __m256i sh = _mm256_setr_epi8(14, 12, 10, 8, 6, 4, 2, 0, -1, -1, -1, -1, -1, -1, -1, -1, 14, 12, 10, 8, 6, 4, 2, 0, -1, -1,
                                        -1, -1, -1, -1, -1, -1);
    const __m256i z = _mm256_shuffle_epi8(x, sh);
    w0 = (uint64_t)_mm256_extract_epi64(z, 0);
    w1 = (uint64_t)_mm256_extract_epi64(z, 2);
}

// 128 two-bit ranks -> four words: per 32-byte vector two multiply-adds leave one finished byte (4 symbols, the first on
// top) in every 32-bit lane; two saturating packs bring the 32 finished bytes of four vectors together, a byte shuffle
// and a lane permutation put them in word order (byte 7 - l of word t = symbols 4 l .. 4 l + 3 of vector t)
static inline __m256i pack128x2(__m256i v0, __m256i v1, __m256i v2, __m256i v3) {
    const __m256i m1 = _mm256_set1_epi16(0x0104), m2 = _mm256_set1_epi32(0x00010010);
    const __m256i y0 = _mm256_madd_epi16(_mm256_maddubs_epi16(v0, m1), m2);
    const __m256i y1 = _mm256_madd_epi16(_mm256_maddubs_epi16(v1, m1), m2);
    const __m256i y2 = _mm256_madd_epi16(_mm256_maddubs_epi16(v2, m1), m2);
    const __m256i y3 = _mm256_madd_epi16(_mm256_maddubs_epi16(v3, m1), m2);
    const __m256i b = _mm256_packus_epi16(_mm256_packus_epi32(y0, y1), _mm256_packus_epi32(y2, y3));
    // low half: symbols 0..15 of vectors 0..3 (4 bytes each), high half: symbols 16..31; reverse every 4-byte group
    const __m256i rev = _mm256_setr_epi8(3, 2, 1, 0, 7, 6, 5, 4, 11, 10, 9, 8, 15, 14, 13, 12, 3, 2, 1, 0, 7, 6, 5, 4, 11, 10, 9, 8,
                                         15, 14, 13, 12);
    const __m256i r = _mm256_shuffle_epi8(b, rev);
    return _mm256_permutevar8x32_epi32(r, _mm256_setr_epi32(4, 0, 5, 1, 6, 2, 7, 3));
}
#endif

template <int BITS>
bool pack_stream_range(const uint8_t *ranks, uint64_t n, uint32_t sigma, uint64_t *words, uint64_t w_lo, uint64_t w_hi) {
    constexpr uint32_t SPW = 64 / BITS;
    constexpr uint32_t CPW = SPW / 8;
    const uint64_t full_hi = std::min<uint64_t>(w_hi, n / SPW);  // words below it are whole
    uint64_t w = w_lo;
    bool bad = false;
#if defined(__AVX2__)
    __m256i vmax = _mm256_setzero_si256();
    if (BITS == 2) {
        for (; w + 4 <= full_hi; w += 4) {
            const __m256i *src = reinterpret_cast<const __m256i *>(ranks + w * 32);
            const __m256i v0 = _mm256_loadu_si256(src), v1 = _mm256_loadu_si256(src + 1), v2 = _mm256_loadu_si256(src + 2),
                          v3 = _mm256_loadu_si256(src + 3);
            vmax = _mm256_max_epu8(_mm256_max_epu8(vmax, _mm256_max_epu8(v0, v1)), _mm256_max_epu8(v2, v3));
            _mm256_storeu_si256(reinterpret_cast<__m256i *>(words + w), pack128x2(v0, v1, v2, v3));
        }
    } else if (BITS == 4) {
        for (; w + 2 <= full_hi; w += 2) {
            const __m256i v = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(ranks + w * 16));
            vmax = _mm256_max_epu8(vmax, v);
            pack32x4(v, words[w], words[w + 1]);
        }
    } else {
        // 8 bits: a word is its 8 ranks with the byte order reversed (symbol 0 on top)
        const __m256i rev = _mm256_setr_epi8(7, 6, 5, 4, 3, 2, 1, 0, 15, 14, 13, 12, 11, 10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 0, 15, 14, 13,
                                             12, 11, 10, 9, 8);
        for (; w + 4 <= full_hi; w += 4) {
            const __m256i v = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(ranks + w * 8));
            vmax = _mm256_max_epu8(vmax, v);
            _mm256_storeu_si256(reinterpret_cast<__m256i *>(words + w), _mm256_shuffle_epi8(v, rev));
        }
    }
    {
        alignas(32) uint8_t mx[32];
        _mm256_store_si256(reinterpret_cast<__m256i *>(mx), vmax);
        for (int j = 0; j < 32; ++j) bad |= mx[j] >= sigma;
    }
#endif
    for (; w < w_hi; ++w) {  // the words the vector loops left, and the one the run ends in: symbol by symbol
        uint64_t acc = 0;
        for (uint32_t c = 0; c < CPW; ++c) {
            uint64_t v = 0;
            for (uint32_t j = 0; j < 8; ++j) {
                const uint64_t s = w * SPW + 8 * c + j;
                if (s < n) {
                    bad |= ranks[s] >= sigma;
                    v |= (uint64_t)ranks[s] << (8 * j);
                }
            }
            acc |= pack8<BITS>(v) << (64 - 8 * BITS * (c + 1));
        }
        words[w] = acc;
    }
    return !bad;
}

}  // namespace

uint64_t pack_stream_words(uint64_t n, uint32_t bits) { return (n + 64 / bits - 1) / (64 / bits); }

bool pack_stream_host(const uint8_t *ranks, uint64_t n, uint32_t bits, uint32_t sigma, uint64_t *words, unsigned part,
                      unsigned n_parts) {
    const uint64_t n_words = pack_stream_words(n, bits);
    // parts are cut at multiples of four words (the vector loop's step)
    const uint64_t quads = (n_words + 3) / 4;
    const uint64_t w_lo = std::min(n_words, quads * part / n_parts * 4), w_hi = std::min(n_words, quads * (part + 1) / n_parts * 4);
    if (bits == 2) return pack_stream_range<2>(ranks, n, sigma, words, w_lo, w_hi);
    if (bits == 4) return pack_stream_range<4>(ranks, n, sigma, words, w_lo, w_hi);
    return pack_stream_range<8>(ranks, n, sigma, words, w_lo, w_hi);
}

}  // namespace kb
