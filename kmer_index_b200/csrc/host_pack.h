// Host-side helpers of the C ABI's host-buffer search (capi.cu): a small persistent thread pool, the query lengths and the
// streaming pack of query batches and texts (1 byte per rank -> the device's b-bit MSB-first words) before they cross PCIe.
#pragma once

#include <cstdint>
#include <functional>

namespace kb {

// Runs fn(i) for i in [0, n_tasks) on the pool's threads; returns a ticket to wait on. One batch at a time.
class HostPool {
  public:
    static HostPool &instance();
    unsigned threads() const;
    void submit(unsigned n_tasks, std::function<void(unsigned)> fn);  // asynchronous
    void wait();                                                       // until the submitted batch is done
    void run(unsigned n_tasks, std::function<void(unsigned)> fn) {
        submit(n_tasks, std::move(fn));
        wait();
    }

  private:
    HostPool();
    ~HostPool();
    struct Impl;
    Impl *impl_;
};

// Queries [q_begin, q_end) of a host batch: lens[i - q_begin] = length (its low 16 bits: valid when the returned longest
// length is below 65 536) and the longest length.
uint64_t query_lengths_host(const uint64_t *q_offsets, uint64_t q_begin, uint64_t q_end, uint16_t *lens, unsigned part,
                            unsigned n_parts);

// Streaming pack of a contiguous run of n ranks, query boundaries ignored: symbol s lands in bits
// [64 - bits (s % spw + 1), 64 - bits (s % spw)) of words[s / spw]; the unused low bits of the last word are zero. The
// device cuts the stream into per-query words afterwards (align_stream_kernel, capi.cu), which costs it ~1 ms per 10^8
// queries -- per-query work on the host cores costs 50x that. `part` of `n_parts`: the slice of the words this call
// writes (pack_stream_words(n, bits) in all). Returns false when a rank >= sigma was seen.
uint64_t pack_stream_words(uint64_t n, uint32_t bits);
bool pack_stream_host(const uint8_t *ranks, uint64_t n, uint32_t bits, uint32_t sigma, uint64_t *words, unsigned part,
                      unsigned n_parts);

}  // namespace kb
