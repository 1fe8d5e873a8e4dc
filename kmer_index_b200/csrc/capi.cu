// C ABI of libkmer_b200.so (include/kmer_b200.h): host-side orchestration of the build and search kernels.
// No CPU fallback anywhere: every computing entry point needs a CUDA device.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <new>
#include <string>
#include <system_error>
#include <thread>
#include <vector>

#include "host_pack.h"
#include "launch.h"
#include "radix.cuh"

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}

#define KB_CUDA(expr)                                                                                      \
    do {                                                                                                   \
        cudaError_t _e = (expr);                                                                           \
        if (_e != cudaSuccess) {                                                                           \
            cudaGetLastError();                                                                            \
            return fail(_e == cudaErrorMemoryAllocation ? KMER_B200_ERR_OUT_OF_MEMORY : KMER_B200_ERR_CUDA, \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                               \
        }                                                                                                  \
    } while (0)

#define KB_TRY(expr)           \
    do {                       \
        int _s = (expr);       \
        if (_s != 0) return _s; \
    } while (0)

// kmer::detail::fast_pow, fast_pow.hpp:46-93
uint64_t fast_pow(uint64_t base, uint8_t exp) {
    if (exp >= 63) return base == 1 ? 1 : 0;  // the "overflow" row of highest_bit_set
    uint64_t result = 1;
    while (exp) {
        if (exp & 1) result *= base;
        exp >>= 1;
        base *= base;
    }
    return result;
}

uint32_t bit_length(uint64_t v) {
    uint32_t b = 0;
    while (v) {
        ++b;
        v >>= 1;
    }
    return b;
}

enum KernelId : int {
    K_PACK_TEXT = 0,
    K_HIST_TEXT,
    K_HIST_PAIRS,
    K_COLUMN_SCAN,
    K_SCATTER_TEXT,
    K_SCATTER_PAIRS,
    K_DIRECTORY_FILL,
    K_SEARCH_COUNT,
    K_SEARCH_WRITE,
    K_SEARCH_PRESENCE,
    K_OFFSETS_SCAN,
    K_SEGMENT_SORT,
    K_APPROX_BEST,
    K_APPROX_SINGLE,
    K_APPROX_DISTANCES,
    K_SEED_COUNT,
    K_SEED_WRITE,
    K_VOTES_COUNT,
    K_VOTES_WRITE,
    K_VOTES_OVERFLOW,
    K_COUNT_
};

const char *const kKernelNames[K_COUNT_] = {
    "pack_text",       "radix_hist_text", "radix_hist_pairs", "column_scan",     "radix_scatter_text", "radix_scatter_pairs",
    "directory_fill",  "search_count",    "search_write",     "search_presence", "offsets_scan",       "segment_sort",
    "approx_best",     "approx_single",   "approx_distances", "seed_count",      "seed_write",         "votes_count",
    "votes_write",     "votes_overflow"};

struct Profiler {
    bool enabled = false;
    cudaStream_t stream = nullptr;
    uint64_t launches[K_COUNT_] = {};
    double bytes[K_COUNT_] = {};
    double ms[K_COUNT_] = {};
    struct Pending {
        int id;
        cudaEvent_t a, b;
    };
    std::vector<Pending> pending;
    std::vector<cudaEvent_t> pool;

    cudaEvent_t get_event() {
        if (!pool.empty()) {
            cudaEvent_t e = pool.back();
            pool.pop_back();
            return e;
        }
        cudaEvent_t e;
        cudaEventCreate(&e);
        return e;
    }
    void begin(int id, double algorithmic_bytes, uint64_t n_launches = 1) {
        launches[id] += n_launches;
        bytes[id] += algorithmic_bytes;
        if (!enabled) return;
        Pending p{id, get_event(), get_event()};
        cudaEventRecord(p.a, stream);
        pending.push_back(p);
    }
    void end() {
        if (!enabled) return;
        cudaEventRecord(pending.back().b, stream);
    }
    void resolve() {
        if (pending.empty()) return;
        cudaStreamSynchronize(stream);
        for (auto &p : pending) {
            float t = 0;
            if (cudaEventElapsedTime(&t, p.a, p.b) == cudaSuccess) ms[p.id] += t;
            pool.push_back(p.a);
            pool.push_back(p.b);
        }
        pending.clear();
    }
    void reset() {
        resolve();
        for (int i = 0; i < K_COUNT_; ++i) {
            launches[i] = 0;
            bytes[i] = 0;
            ms[i] = 0;
        }
    }
    ~Profiler() {
        resolve();
        for (auto e : pool) cudaEventDestroy(e);
    }
};

struct HostElement {
    kb::Element dev{};  // device pointers inside
    uint32_t key_bits = 0;
    uint32_t sort_passes = 0;
    uint64_t bytes = 0;
    uint32_t *d_dir = nullptr, *d_pos = nullptr;
    void *d_keys = nullptr;  // uint32_t or uint64_t hashes (key_bytes); null for a dense directory
    uint32_t key_bytes = 4;
    uint64_t n_occupied = 0;  // distinct hashes (non-empty buckets), measured on first use by kmer_b200_plan_table
    int adopted = 0;         // 1: pos / dir belong to the caller (kmer_b200_adopt_element); 2: assembled by the library, owned
    bool view = false;       // shared-positions index: no arrays of its own, a prefix view of the largest k's (kb::Element::width)
    bool in_parts = false;   // peer-positions index: the positions stay in the caller's per-GPU parts (kb::Element::pos_part)
};

// Shared-positions multi-k index (kmer_b200_config::reserved bit 1): every element but the one with the largest k becomes
// a view of that one's arrays. `owner` must be built (or loaded).
void make_view(HostElement &he, const HostElement &owner, uint32_t k, uint32_t sigma) {
    he = HostElement{};
    he.view = true;
    he.dev = owner.dev;  // dir / keys / pos / shift / n_kmers / key_space / key_bytes are the owner's
    he.dev.k = k;
    he.dev.k_phys = owner.dev.k;
    he.dev.width = fast_pow(sigma, (uint8_t)(owner.dev.k - k));
    he.key_bits = std::max<uint32_t>(1, bit_length(fast_pow(sigma, (uint8_t)k) - 1));
    he.key_bytes = owner.key_bytes;
    he.sort_passes = 0;
    he.bytes = 0;
}

// the hash range element `k` of this index covers: all of [0, sigma^k), or one of cfg.key_parts equal slices
struct KeyRange {
    uint64_t lo, hi;
};
KeyRange key_range_of(const kmer_b200_config &cfg, uint64_t key_space) {
    if (cfg.key_parts <= 1) return KeyRange{0, key_space};
    uint64_t width = (key_space + cfg.key_parts - 1) / cfg.key_parts;
    width = (width + 63) / 64 * 64;
    const uint64_t lo = std::min<uint64_t>((uint64_t)cfg.key_part * width, key_space);
    return KeyRange{lo, std::min<uint64_t>(lo + width, key_space)};
}

}  // namespace

struct kmer_b200_index {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_in = nullptr, copy_out = nullptr;  // host-batch pipeline: H2D / D2H engines next to `stream`
    cudaStream_t copy_in2 = nullptr;                     // second H2D queue (raw chunks of search_batch_host_chunked)
    kmer_b200_config cfg{};
    uint64_t n = 0;
    uint32_t sigma = 0, bits = 0;
    std::vector<uint32_t> ks;
    std::vector<HostElement> elems;
    uint64_t *d_text = nullptr;
    uint64_t text_words = 0;
    // scheme tables (host copies for kmer_b200_scheme + device copies)
    std::vector<uint32_t> sum_off;
    std::vector<uint8_t> sum_elem, use_multi;
    uint32_t *d_sum_off = nullptr;
    uint8_t *d_sum_elem = nullptr, *d_use_multi = nullptr;
    kb::DeviceIndex host_index{};
    kb::DeviceIndex *d_index = nullptr;
    uint32_t *d_flags = nullptr;     // u32[4]: error bits, unsorted-segment count, u64 mask of sub-k lengths w/o aux
    uint64_t *h_pinned = nullptr;    // small pinned scratch: [0] total hits, [1] flags, [2] max len, [3] gathers
    unsigned long long *d_gathers = nullptr;  // profile mode: sectors gathered by the last search
    uint64_t last_gathers = 0;
    uint64_t last_h2d = 0, last_d2h = 0;  // bytes the last host-buffer search moved over PCIe (kmer_b200_last_search_transfer)
    uint64_t build_h2d = 0;               // bytes the text took on its way to the device (kmer_b200_build_transfer)
    uint32_t last_host_path = 0, last_raw_pct = 0;  // which host pipeline it took (kmer_b200_last_search_host_path)
    double last_pack_gbs = 0;
    uint32_t host_sharers = 1;  // devices of a multi-device handle searching at the same time: they share the host packers
    uint64_t device_bytes = 0;
    bool reaches_end = true;  // the local slice ends at the end of the whole text
    bool sharded = false;
    double max_avg_bucket = 0;  // max over elements of (k-mers / distinct possible hashes)
    Profiler prof;
    std::mutex mu;  // serialises searches on one handle (they share the stream and the flag words)
    size_t h_pinned_cap = 0;
    // a multi-device handle (cfg.n_devices > 1) owns one whole index per device and nothing else
    std::vector<kmer_b200_index *> replicas;
    // collection index (kmer_b200_attach_records): the record table starts[0..R] (host and device) and the boundary
    // bitmap of DeviceIndex::boundary; empty / null otherwise
    std::vector<uint64_t> starts;
    uint64_t *d_starts = nullptr;
    uint64_t *d_boundary = nullptr;
};

static inline kmer_b200_index *primary(kmer_b200_index *ix) { return (ix && !ix->replicas.empty()) ? ix->replicas[0] : ix; }
static inline const kmer_b200_index *primary(const kmer_b200_index *ix) { return (ix && !ix->replicas.empty()) ? ix->replicas[0] : ix; }

struct kmer_b200_result {
    kmer_b200_index *index = nullptr;
    bool on_device = false;
    uint64_t n_queries = 0, n_positions = 0;
    uint64_t *offsets = nullptr;
    uint32_t *positions = nullptr;
    uint8_t *status = nullptr;
    uint32_t *hit_queries = nullptr;  // device results: [0] = n, [1..n] = ids of the queries the count pass found hits for
    uint8_t *distances = nullptr;      // approximate search with KMER_B200_APPROX_DISTANCES: d(p) per position, or null
    uint8_t *best_distance = nullptr;  // approximate search, hit strategies other than "all": d_min per query, or null
    uint32_t *seed_offsets = nullptr;  // seeding: the query offset j of each position, or null
    uint32_t *kmer_counts = nullptr;   // seeding: the occurrence count of each k-mer of the batch, or null
    uint32_t *votes = nullptr;         // record votes (positions hold the records): the votes of each entry, or null
    uint32_t *kmer_hits = nullptr;     // record votes: the counted k-mers of each query, or null
    uint64_t n_kmers = 0;
    size_t cap_offsets = 0, cap_positions = 0, cap_status = 0;  // host buffers: byte capacities
    size_t cap_distances = 0, cap_best_distance = 0, cap_seed_offsets = 0, cap_kmer_counts = 0;
    size_t cap_votes = 0, cap_kmer_hits = 0;
    bool positions_pageable = false;  // very large position lists live in plain malloc memory
};

namespace {

// Every array a result can hold: f(array member, capacity member of its host buffer, element count). The one list that
// kmer_b200_result_free and result_to_host walk; hit_queries lives on the device only (no capacity).
template <typename F>
void for_each_result_array(const kmer_b200_result &r, F &&f) {
    using R = kmer_b200_result;
    const uint64_t Q = r.n_queries, P = r.n_positions;
    f(&R::offsets, &R::cap_offsets, Q + 1);
    f(&R::status, &R::cap_status, Q);
    f(&R::positions, &R::cap_positions, P);
    f(&R::distances, &R::cap_distances, P);
    f(&R::best_distance, &R::cap_best_distance, Q);
    f(&R::seed_offsets, &R::cap_seed_offsets, P);
    f(&R::kmer_counts, &R::cap_kmer_counts, r.n_kmers);
    f(&R::votes, &R::cap_votes, P);
    f(&R::kmer_hits, &R::cap_kmer_hits, Q);
    f(&R::hit_queries, (size_t R::*)nullptr, Q + 1);
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// ---- guarded allocations (debug aid; compute-sanitizer is not available on every pool) ------------------------------
// KMER_B200_GUARD=1: every device allocation of the library is bracketed by two 4 KB zones filled with a canary byte,
// and the zones are verified on the device when the allocation is freed. A store that lands up to 4 KB before or behind
// any buffer -- scatter destinations, result lists, staging rings -- is counted; kmer_b200_debug_guard_violations()
// returns the count. Reads are not covered. Off by default: no cost.
constexpr size_t kGuardBytes = 4096;
constexpr int kGuardByte = 0xA5;
bool guard_mode() {
    static const bool on = [] {
        const char *e = std::getenv("KMER_B200_GUARD");
        return e && std::atoi(e) != 0;
    }();
    return on;
}
std::mutex g_guard_mu;
std::unordered_map<void *, size_t> g_guard_sizes;     // user pointer -> user bytes
unsigned long long *g_guard_bad = nullptr;             // pinned, mapped: damaged canary bytes seen so far

__global__ void __launch_bounds__(256) guard_check_kernel(const uint8_t *__restrict__ base, size_t user_bytes,
                                                          unsigned long long *bad) {
    unsigned n = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * kGuardBytes; i += (size_t)gridDim.x * blockDim.x) {
        const size_t at = i < kGuardBytes ? i : kGuardBytes + user_bytes + (i - kGuardBytes);
        n += base[at] != (uint8_t)kGuardByte;
    }
    if (n) atomicAdd_system(bad, (unsigned long long)n);
}

cudaError_t kb_malloc_async(void **p, size_t bytes, cudaStream_t st) {
    if (!guard_mode()) return cudaMallocAsync(p, bytes, st);
    uint8_t *base = nullptr;
    cudaError_t e = cudaMallocAsync((void **)&base, bytes + 2 * kGuardBytes, st);
    if (e != cudaSuccess) return e;
    cudaMemsetAsync(base, kGuardByte, kGuardBytes, st);
    cudaMemsetAsync(base + kGuardBytes + bytes, kGuardByte, kGuardBytes, st);
    *p = base + kGuardBytes;
    std::lock_guard<std::mutex> lock(g_guard_mu);
    if (!g_guard_bad) {
        cudaHostAlloc((void **)&g_guard_bad, sizeof(unsigned long long), cudaHostAllocMapped | cudaHostAllocPortable);
        if (g_guard_bad) *g_guard_bad = 0;
    }
    g_guard_sizes[*p] = bytes;
    return cudaSuccess;
}

void kb_free_async(void *p, cudaStream_t st) {
    if (!p) return;
    if (!guard_mode()) {
        cudaFreeAsync(p, st);
        return;
    }
    size_t bytes = 0;
    bool known = false;
    {
        std::lock_guard<std::mutex> lock(g_guard_mu);
        auto it = g_guard_sizes.find(p);
        if (it != g_guard_sizes.end()) {
            known = true;
            bytes = it->second;
            g_guard_sizes.erase(it);
        }
    }
    if (!known) {  // not ours (never happens for pointers this file allocates)
        cudaFreeAsync(p, st);
        return;
    }
    uint8_t *base = (uint8_t *)p - kGuardBytes;
    if (g_guard_bad) guard_check_kernel<<<8, 256, 0, st>>>(base, bytes, g_guard_bad);
    cudaFreeAsync(base, st);
}

template <typename T>
int dev_alloc(kmer_b200_index *ix, T **p, uint64_t count, bool persistent) {
    const size_t bytes = std::max<uint64_t>(count, 1) * sizeof(T);
    KB_CUDA(kb_malloc_async((void **)p, bytes, ix->stream));
    if (persistent) ix->device_bytes += bytes;
    return 0;
}

template <typename T>
void dev_free(kmer_b200_index *ix, T *p) {
    if (p) kb_free_async((void *)p, ix->stream);
}

// Process-wide cache of pinned host buffers (results handed to the caller, small scratch words). Pinned
// allocation costs milliseconds, so buffers outlive the index that first asked for them.
std::mutex g_pinned_mu;
std::vector<std::pair<void *, size_t>> g_pinned_cache;

void *pinned_get(size_t bytes, size_t *cap) {
    bytes = std::max<size_t>(bytes, 64);
    {
        std::lock_guard<std::mutex> lock(g_pinned_mu);
        size_t best = SIZE_MAX, best_i = SIZE_MAX;
        for (size_t i = 0; i < g_pinned_cache.size(); ++i) {
            const size_t c = g_pinned_cache[i].second;
            if (c >= bytes && c < best) {
                best = c;
                best_i = i;
            }
        }
        if (best_i != SIZE_MAX && best <= 4 * bytes + (1u << 20)) {
            void *p = g_pinned_cache[best_i].first;
            g_pinned_cache.erase(g_pinned_cache.begin() + best_i);
            *cap = best;
            return p;
        }
    }
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    *cap = bytes;
    return p;
}

void pinned_put(void *p, size_t cap) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> lock(g_pinned_mu);
        if (g_pinned_cache.size() < 32) {
            g_pinned_cache.emplace_back(p, cap);
            return;
        }
    }
    cudaFreeHost(p);
}

// choose_search_scheme, kmer_index.hpp:407-476, in integer arithmetic.
// sum lists are stored as chains (last summand + previous length) and flattened at the end.
struct SchemeHost {
    std::vector<uint32_t> ks;  // template order
    std::vector<uint32_t> sum_off;
    std::vector<uint8_t> sum_elem, use_multi;
};

void build_scheme(SchemeHost *ix) {
    const uint32_t R = kb::kQuerySizeRange;
    std::vector<uint32_t> all_ks(ix->ks);
    std::sort(all_ks.begin(), all_ks.end(), [](uint32_t a, uint32_t b) { return a > b; });  // :410
    std::vector<uint32_t> high;
    for (uint32_t k : all_ks)
        if (k >= 9) high.push_back(k);  // :414
    std::vector<uint32_t> len(R, 0), last(R, 0), prev(R, 0);
    ix->use_multi.assign(R, 0);
    for (uint32_t k : high)  // :421-425
        if (k < R) {
            len[k] = 1;
            last[k] = k;
            ix->use_multi[k] = 1;
        }
    for (uint32_t q = all_ks.front() + 1; q < R; ++q)  // :427-443: first (largest) high k whose remainder is reachable
        for (uint32_t k : high)
            if (len[q - k] != 0) {
                len[q] = len[q - k] + 1;
                last[q] = k;
                prev[q] = q - k;
                ix->use_multi[q] = 1;
                break;
            }
    for (uint32_t q = 0; q < R; ++q) {  // :445-475
        if (len[q] != 0) continue;
        uint32_t best = all_ks.front();
        if (q < all_ks.front()) {
            // smallest k >= q (:450-462)
            for (uint32_t k : all_ks)
                if (q <= k && k - q < best - q) best = k;
        } else {
            // k minimising the padding ceil(q/k)*k - q; ties keep the larger k (:463-474)
            auto waste = [q](uint32_t k) { return ((q + k - 1) / k) * k - q; };
            for (uint32_t k : all_ks)
                if (waste(k) < waste(best)) best = k;
        }
        len[q] = 1;
        last[q] = best;
    }
    auto elem_of = [ix](uint32_t k) {
        for (size_t i = 0; i < ix->ks.size(); ++i)
            if (ix->ks[i] == k) return (uint8_t)i;
        return (uint8_t)0;
    };
    ix->sum_off.assign(R + 2, 0);
    uint64_t total = 0;
    for (uint32_t q = 0; q < R; ++q) {
        ix->sum_off[q] = (uint32_t)total;
        total += len[q];
    }
    ix->sum_off[R] = (uint32_t)total;
    ix->sum_off[R + 1] = (uint32_t)total;
    ix->sum_elem.assign(total, 0);
    for (uint32_t q = 0; q < R; ++q) {
        uint64_t o = (uint64_t)ix->sum_off[q] + len[q];
        uint32_t c = q;
        for (uint32_t j = 0; j < len[q]; ++j) {
            ix->sum_elem[--o] = elem_of(last[c]);
            c = prev[c];
        }
    }
}

// Sorters: both leave he.d_keys (sorted hashes) and he.d_pos (positions stably sorted by hash).
// (a) tiled LSD sort: per-tile histograms + column scan + scatter per pass, (hash, position) in separate arrays.
//     Used for 64-bit hashes and k-mers wider than one packed window.
int sort_element_tiled(kmer_b200_index *ix, uint32_t k, HostElement &he, uint32_t digit_bits, KeyRange part, uint64_t *n_sorted) {
    using namespace kb;
    cudaStream_t st = ix->stream;
    Profiler &pf = ix->prof;
    const uint64_t n_text_kmers = ix->n - k + 1;
    const uint32_t key_bytes = he.key_bytes;
    const bool partial = part.lo != 0 || part.hi != fast_pow(ix->sigma, (uint8_t)k);
    PackedText text{ix->d_text, ix->n, ix->bits, ix->sigma};
    // a key-range part: the text is first filtered into the (hash - lo, position) pairs of the part, in position order
    uint64_t n_kmers = n_text_kmers;
    uint32_t sort_bits = he.key_bits;
    void *f_keys = nullptr;
    uint32_t *f_vals = nullptr;
    if (partial) {
        const uint32_t ft = filter_tiles(n_text_kmers);
        uint64_t *tile_counts = nullptr, *block_sums = nullptr;
        KB_TRY(dev_alloc(ix, &tile_counts, (uint64_t)ft + 1, false));
        KB_TRY(dev_alloc(ix, &block_sums, offsets_scan_blocks(ft) + 1, false));
        pf.begin(K_HIST_TEXT, (double)n_text_kmers * ix->bits / 8.0);
        launch_owned_count(text, k, n_text_kmers, part.lo, part.hi, tile_counts, st);
        pf.end();
        launch_offsets_scan(tile_counts, ft, block_sums, st);
        KB_CUDA(cudaMemcpyAsync(&ix->h_pinned[6], tile_counts + ft, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        n_kmers = ix->h_pinned[6];
        KB_TRY(dev_alloc(ix, (uint8_t **)&f_keys, std::max<uint64_t>(n_kmers, 1) * key_bytes, true));
        KB_TRY(dev_alloc(ix, &f_vals, std::max<uint64_t>(n_kmers, 1), true));
        pf.begin(K_SCATTER_TEXT, (double)n_text_kmers * ix->bits / 8.0 + 8.0 * n_kmers);
        launch_owned_write(text, k, n_text_kmers, part.lo, part.hi, tile_counts, (uint32_t *)f_keys, f_vals, st);
        pf.end();
        dev_free(ix, tile_counts);
        dev_free(ix, block_sums);
        sort_bits = std::max<uint32_t>(1, bit_length(part.hi - part.lo - 1));
    }
    *n_sorted = n_kmers;
    he.sort_passes = (sort_bits + digit_bits - 1) / digit_bits;
    const uint32_t bits_per_pass = (sort_bits + he.sort_passes - 1) / he.sort_passes;
    const uint32_t mask = (1u << bits_per_pass) - 1;
    const uint32_t n_tiles = (uint32_t)((n_kmers + sort_tile_size() - 1) / sort_tile_size());
    const uint32_t n_chunks = (n_tiles + scan_chunk_tiles() - 1) / scan_chunk_tiles();
    const double text_bytes = (double)n_kmers * ix->bits / 8.0;
    const double hist_bytes = (double)n_tiles * kRadix * 4;
    void *keys[2] = {nullptr, nullptr};
    uint32_t *vals[2] = {nullptr, nullptr};
    uint32_t *tile_hist = nullptr, *chunk_sums = nullptr;
    auto alloc_keys = [&](void **p) { return dev_alloc(ix, (uint8_t **)p, std::max<uint64_t>(n_kmers, 1) * key_bytes, true); };
    KB_TRY(dev_alloc(ix, &tile_hist, (uint64_t)std::max(n_tiles, 1u) * kRadix, false));
    KB_TRY(dev_alloc(ix, &chunk_sums, (uint64_t)std::max(n_chunks, 1u) * kRadix, false));
    int cur = 0;
    uint32_t first_pair_pass = 1;
    if (partial) {
        keys[0] = f_keys;  // every pass runs over the filtered pairs
        vals[0] = f_vals;
        first_pair_pass = 0;
    } else {
        KB_TRY(alloc_keys(&keys[0]));
        KB_TRY(dev_alloc(ix, &vals[0], n_kmers, true));
        // pass 0: keys come straight from the packed text
        pf.begin(K_HIST_TEXT, text_bytes + hist_bytes);
        launch_hist_text(text, k, n_kmers, 0, mask, tile_hist, st);
        pf.end();
        pf.begin(K_COLUMN_SCAN, 3 * hist_bytes, 3);
        launch_column_scan(tile_hist, n_tiles, chunk_sums, st);
        pf.end();
        pf.begin(K_SCATTER_TEXT, text_bytes + hist_bytes + (4.0 + key_bytes) * n_kmers);
        launch_scatter_text(text, k, key_bytes, n_kmers, 0, mask, tile_hist, keys[0], vals[0], st);
        pf.end();
    }
    for (uint32_t p = first_pair_pass; p < he.sort_passes && n_kmers > 0; ++p) {
        const int nxt = cur ^ 1;
        if (!keys[nxt]) {
            KB_TRY(alloc_keys(&keys[nxt]));
            KB_TRY(dev_alloc(ix, &vals[nxt], n_kmers, true));
        }
        const uint32_t shift = p * bits_per_pass;
        pf.begin(K_HIST_PAIRS, (double)key_bytes * n_kmers + hist_bytes);
        launch_hist_pairs(keys[cur], key_bytes, n_kmers, shift, mask, tile_hist, st);
        pf.end();
        pf.begin(K_COLUMN_SCAN, 3 * hist_bytes, 3);
        launch_column_scan(tile_hist, n_tiles, chunk_sums, st);
        pf.end();
        pf.begin(K_SCATTER_PAIRS, 2.0 * (4.0 + key_bytes) * n_kmers + hist_bytes);
        launch_scatter_pairs(keys[cur], vals[cur], key_bytes, n_kmers, shift, mask, tile_hist, keys[nxt], vals[nxt], st);
        pf.end();
        cur = nxt;
    }
    KB_CUDA(cudaGetLastError());
    if (keys[cur ^ 1]) {
        dev_free(ix, (uint8_t *)keys[cur ^ 1]);
        dev_free(ix, vals[cur ^ 1]);
        ix->device_bytes -= std::max<uint64_t>(n_kmers, 1) * (sizeof(uint32_t) + key_bytes);
    }
    dev_free(ix, tile_hist);
    dev_free(ix, chunk_sums);
    he.d_keys = keys[cur];
    he.d_pos = vals[cur];
    return 0;
}

// (b) single-sweep sort (onesweep.cu): 32-bit hashes. All digit histograms up front from the text, then one scatter
//     kernel per pass (bulk-copy tile loads, decoupled look-back, 8-byte (hash, position) records between passes).
int sort_element_onesweep(kmer_b200_index *ix, uint32_t k, HostElement &he, uint32_t digit_bits, uint64_t *n_sorted) {
    using namespace kb;
    cudaStream_t st = ix->stream;
    Profiler &pf = ix->prof;
    const uint64_t n_kmers = ix->n - k + 1;
    PackedText text{ix->d_text, ix->n, ix->bits, ix->sigma};
    // digit width: equal shares of the hash bits; for a power-of-two alphabet a whole number of symbols, so that a
    // digit is a c-mer of the text and one c-mer histogram yields every pass's digit histogram
    const bool pow2 = ix->sigma == (1u << ix->bits);
    uint32_t passes = (he.key_bits + digit_bits - 1) / digit_bits;
    uint32_t w = (he.key_bits + passes - 1) / passes;
    if (pow2) {
        w = (w + ix->bits - 1) / ix->bits * ix->bits;
        if (w > (uint32_t)kRadixBitsMax) w = kRadixBitsMax / ix->bits * ix->bits;
        passes = (he.key_bits + w - 1) / w;
    }
    if (passes > 8) return fail(KMER_B200_ERR_UNSUPPORTED, "more than 8 digit passes");
    he.sort_passes = passes;
    const uint32_t mask = (1u << w) - 1;
    const uint32_t n_tiles = (uint32_t)((n_kmers + sort_tile_size() - 1) / sort_tile_size());
    const double text_bytes = (double)n_kmers * ix->bits / 8.0;
    const double status_bytes = 2.0 * (double)n_tiles * kRadix * 8;  // aggregate + inclusive word per (tile, digit)

    uint64_t *status = nullptr;
    uint32_t *scratch = nullptr;  // [0, 2048): histogram scratch, [2048, 4096): digit bases, [4096, 4104): tile counters
    uint2 *pairs[2] = {nullptr, nullptr};
    uint32_t *keys = nullptr, *pos = nullptr;
    auto cleanup = [&](int code) {
        dev_free(ix, status);
        dev_free(ix, scratch);
        dev_free(ix, pairs[0]);
        dev_free(ix, pairs[1]);
        if (code != 0) {
            dev_free(ix, keys);
            dev_free(ix, pos);
        }
        return code;
    };
    if (dev_alloc(ix, &status, (uint64_t)n_tiles * kRadix, false) || dev_alloc(ix, &scratch, 4096 + 8, false))
        return cleanup(KMER_B200_ERR_OUT_OF_MEMORY);
    cudaMemsetAsync(status, 0, (uint64_t)n_tiles * kRadix * sizeof(uint64_t), st);
    cudaMemsetAsync(scratch + 4096, 0, 8 * sizeof(uint32_t), st);
    uint32_t *digit_base = scratch + 2048, *counters = scratch + 4096;

    pf.begin(K_HIST_TEXT, text_bytes, 2);
    launch_digit_histograms(text, k, n_kmers, passes, w, he.key_bits, pow2, scratch, digit_base, st);
    pf.end();

    int cur = -1;
    for (uint32_t p = 0; p < passes; ++p) {
        const bool last = p + 1 == passes;
        uint2 *out_pairs = nullptr;
        if (last) {
            // the buffer that is neither read nor written by this pass goes first: the peak stays at two pair buffers
            if (cur >= 0 && pairs[cur ^ 1]) {
                dev_free(ix, pairs[cur ^ 1]);
                pairs[cur ^ 1] = nullptr;
            }
            if (dev_alloc(ix, &pos, n_kmers, true) || dev_alloc(ix, &keys, n_kmers, true)) return cleanup(KMER_B200_ERR_OUT_OF_MEMORY);
        } else {
            const int nxt = cur < 0 ? 0 : cur ^ 1;
            if (!pairs[nxt] && dev_alloc(ix, &pairs[nxt], n_kmers + 2, false)) return cleanup(KMER_B200_ERR_OUT_OF_MEMORY);
            out_pairs = pairs[nxt];
        }
        const double out_bytes = last ? 8.0 * n_kmers : 8.0 * n_kmers;
        if (p == 0) {
            pf.begin(K_SCATTER_TEXT, text_bytes + out_bytes + status_bytes);
            launch_onesweep_pass(&text, k, nullptr, n_kmers, 0, mask, 1, digit_base, status, counters, out_pairs, keys, pos, st);
        } else {
            pf.begin(K_SCATTER_PAIRS, 8.0 * n_kmers + out_bytes + status_bytes);
            launch_onesweep_pass(nullptr, k, pairs[cur], n_kmers, p * w, mask, p + 1, digit_base + p * kRadix, status, counters + p,
                                 out_pairs, keys, pos, st);
        }
        pf.end();
        if (!last) cur = cur < 0 ? 0 : cur ^ 1;
    }
    KB_CUDA(cudaGetLastError());
    he.d_keys = keys;
    he.d_pos = pos;
    *n_sorted = n_kmers;
    return cleanup(0);
}

int build_element(kmer_b200_index *ix, uint32_t k, HostElement &he, bool auxiliary = false) {
    using namespace kb;
    cudaStream_t st = ix->stream;
    Profiler &pf = ix->prof;
    const uint64_t n_kmers = ix->n - k + 1;
    const uint64_t key_space = fast_pow(ix->sigma, (uint8_t)k);
    he.key_bits = std::max<uint32_t>(1, bit_length(key_space - 1));
    uint32_t digit_bits = kRadixBitsMax;
    if (const char *env = std::getenv("KMER_B200_DIGIT_BITS")) {  // tuning experiment: narrower digits, more passes
        const int b = std::atoi(env);
        if (b >= 4 && b <= kRadixBitsMax) digit_bits = (uint32_t)b;
    }
    // 32-bit hashes while sigma^k <= 2^32 (all BASELINE configs), 64-bit above
    const uint32_t key_bytes = he.key_bits > 32 ? 8 : 4;
    he.key_bytes = key_bytes;
    const KeyRange part = key_range_of(ix->cfg, key_space);
    const bool partial = ix->cfg.key_parts > 1;
    if (partial && (key_bytes != 4 || k * ix->bits > 64))
        return fail(KMER_B200_ERR_UNSUPPORTED, "key-range parts need 32-bit hashes (sigma^k <= 2^32)");
    // directory and sorted hashes are relative to part.lo; max_rel = the largest relative hash (2^64 - 1 when sigma^k
    // "overflows" to 0 in fast_pow, i.e. sigma = 2, k = 63)
    const uint64_t max_rel = (partial ? part.hi - part.lo : key_space) - 1;
    uint64_t n_part = n_kmers;                       // k-mers in the part
    const char *sorter = std::getenv("KMER_B200_SORT");  // "onesweep": the single-sweep experiment (DESIGN.md section 4)
    if (!partial && key_bytes == 4 && k * ix->bits <= 64 && sorter && std::strcmp(sorter, "onesweep") == 0) {
        KB_TRY(sort_element_onesweep(ix, k, he, digit_bits, &n_part));
    } else {
        KB_TRY(sort_element_tiled(ix, k, he, digit_bits, part, &n_part));
    }

    // directory: dense (shift 0) while the key space is at most ~4x the number of k-mers -- or whenever it is affordable:
    // a position-range shard (or a key-range part) holds 1/N of the k-mers but must not answer most lookups with a
    // binary search in the sorted hashes just because of that
    uint32_t shift = 0;
    const uint32_t part_bits = std::max<uint32_t>(1, bit_length(max_rel));
    if (ix->cfg.directory_bits) {
        if (part_bits > ix->cfg.directory_bits) shift = part_bits - ix->cfg.directory_bits;
    } else {
        uint32_t want = bit_length(n_part) + 1;
        if (want < 16) want = 16;
        if (part_bits > want) {
            size_t free_b = 0, total_b = 0;
            cudaMemGetInfo(&free_b, &total_b);
            const bool affordable = (ix->sharded || partial) && max_rel < (1ull << 33) && max_rel * 4ull + (1ull << 30) < free_b / 3;
            if (!affordable) shift = part_bits - want;
        }
    }
    if (partial && shift != 0) return fail(KMER_B200_ERR_UNSUPPORTED, "key-range parts need a dense directory");
    if (part_bits > 32 + shift) shift = part_bits - 32;  // directory indices stay below 2^32
    const uint64_t dir_entries = (max_rel >> shift) + 2;
    KB_TRY(dev_alloc(ix, &he.d_dir, dir_entries, true));
    pf.begin(K_DIRECTORY_FILL, (double)key_bytes * n_part + 4.0 * dir_entries);
    launch_directory_fill(he.d_keys, key_bytes, n_part, shift, dir_entries, he.d_dir, st);
    pf.end();
    KB_CUDA(cudaGetLastError());
    if (shift == 0) {
        // dense directory: at(h) is [dir[h], dir[h + 1]) and nothing reads the sorted hashes again (the one place that
        // wants a hash of an entry, the sub-k slab check, recomputes it from the text): 4 bytes per k-mer of HBM back
        dev_free(ix, (uint8_t *)he.d_keys);
        he.d_keys = nullptr;
        ix->device_bytes -= std::max<uint64_t>(n_part, 1) * key_bytes;
    }

    he.dev.k = k;
    he.dev.shift = shift;
    he.dev.n_kmers = n_part;
    he.dev.dir_entries = dir_entries;
    he.dev.key_space = key_space;
    he.dev.dir = he.d_dir;
    he.dev.keys = he.d_keys;
    he.dev.pos = he.d_pos;
    he.dev.key_bytes = key_bytes;
    he.dev.key_lo = partial ? part.lo : 0;
    he.dev.key_hi = partial ? part.hi : UINT64_MAX;
    he.dev.k_phys = k;
    he.dev.width = 1;
    he.bytes = n_part * (sizeof(uint32_t) + (he.d_keys ? key_bytes : 0)) + dir_entries * sizeof(uint32_t);
    if (!auxiliary)
        ix->max_avg_bucket = std::max(ix->max_avg_bucket, (double)n_kmers / (double)std::min<uint64_t>(key_space, n_kmers));
    return 0;
}

#define KB_CUDA_RET(expr)                                                                           \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            cudaGetLastError();                                                                     \
            return fail(_e == cudaErrorMemoryAllocation ? KMER_B200_ERR_OUT_OF_MEMORY : KMER_B200_ERR_CUDA, \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                        \
        }                                                                                           \
    } while (0)

// Validated, empty index: configuration, device, stream, scratch. The caller destroys it on later failures.
int new_index(uint64_t n, uint32_t sigma, const uint32_t *ks, uint32_t n_ks, const kmer_b200_config *cfg_in,
              kmer_b200_index **out) {
    *out = nullptr;
    if (!ks) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "ks is null");
    if (n_ks == 0 || n_ks > (uint32_t)kb::kMaxElements)
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "number of ks must be in [1, 32]");
    if (sigma < 2 || sigma > 256) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "sigma must be in [2, 256]");
    const uint32_t bits = sigma <= 4 ? 2 : (sigma <= 16 ? 4 : 8);
    uint32_t k_max = 0;
    for (uint32_t i = 0; i < n_ks; ++i) {
        const uint32_t k = ks[i];
        // static_assert(k > 0 and k < 64 / log2(sigma)), kmer_index.hpp:42-43
        if (k == 0 || !((double)k < 64.0 / std::log2((double)sigma)))
            return fail(KMER_B200_ERR_INVALID_ARGUMENT, "k must satisfy 0 < k < 64 / log2(sigma) (kmer_index.hpp:42)");
        for (uint32_t j = 0; j < i; ++j)
            if (ks[j] == k) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "duplicate k");
        k_max = std::max(k_max, k);
    }
    if (n < k_max) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "text shorter than the largest k");
    // assert(i + k - 1 < numeric_limits<position_t>::max()), kmer_index.hpp:169 with position_t = uint32_t (:575)
    kmer_b200_config cfg;
    if (cfg_in)
        cfg = *cfg_in;
    else
        kmer_b200_config_default(&cfg);
    const uint64_t n_total = cfg.n_total ? cfg.n_total : n;
    if (cfg.shard_begin + n > n_total) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "shard exceeds n_total");
    if (n_total >= 0xFFFFFFFFull) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "text too large for 32-bit positions");
    const bool sharded = cfg.n_total != 0 && (cfg.shard_begin != 0 || n != n_total);
    const bool reaches_end = cfg.shard_begin + n == n_total;  // the slice ends where the text ends
    if (cfg.halo >= n && cfg.halo) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "halo must be smaller than the slice");
    if (sharded && !reaches_end && cfg.halo + 1 < k_max)
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "interior shards need halo >= max k - 1");

    if (cfg.key_parts > 1 && cfg.key_part >= cfg.key_parts) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "key_part must be < key_parts");
    if (cfg.key_parts > 1 && sharded) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "key-range parts index the whole text: no position-range shard");
    if ((cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS) && n_ks > 1) {
        if (sharded || cfg.key_parts > 1 || cfg.n_devices > 1)
            return fail(KMER_B200_ERR_UNSUPPORTED, "a shared-positions index is unsharded and lives on one device");
        cfg.reserved |= KMER_B200_FLAG_NO_AUX;  // the point is one position array: no per-length copies on demand
    } else {
        cfg.reserved &= ~(uint32_t)KMER_B200_FLAG_SHARED_POSITIONS;
    }
    int device = cfg.device;
    if (device < 0) {
        cudaError_t e = cudaGetDevice(&device);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(KMER_B200_ERR_CUDA, std::string("cudaGetDevice: ") + cudaGetErrorString(e));
        }
    }
    {
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || device >= count) {
            cudaGetLastError();
            return fail(KMER_B200_ERR_CUDA, "no usable CUDA device (libkmer_b200 has no CPU fallback)");
        }
    }
    DeviceGuard guard(device);
    kmer_b200_index *ix = new (std::nothrow) kmer_b200_index();
    if (!ix) return fail(KMER_B200_ERR_OUT_OF_MEMORY, "host allocation failed");
    ix->device = device;
    ix->cfg = cfg;
    ix->n = n;
    ix->sigma = sigma;
    ix->bits = bits;
    ix->ks.assign(ks, ks + n_ks);
    ix->reaches_end = reaches_end;
    ix->sharded = sharded;
    *out = ix;  // from here on the caller owns (and destroys) it
    if (cfg.stream) {
        ix->stream = (cudaStream_t)cfg.stream;
    } else {
        KB_CUDA_RET(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking));
        ix->own_stream = true;
    }
    ix->prof.enabled = cfg.profile != 0;
    ix->prof.stream = ix->stream;
    {
        // keep freed blocks in the stream-ordered pool so repeated builds/searches do not hit the driver
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t threshold = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
        }
    }
    ix->h_pinned = (uint64_t *)pinned_get(8 * sizeof(uint64_t), &ix->h_pinned_cap);
    if (!ix->h_pinned) return fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed");
    KB_TRY(dev_alloc(ix, &ix->d_flags, 4, true));
    KB_TRY(dev_alloc(ix, &ix->d_gathers, 1, true));
    KB_CUDA_RET(cudaMemsetAsync(ix->d_flags, 0, 4 * sizeof(uint32_t), ix->stream));
    ix->text_words = (n * bits + 63) / 64 + 2;
    KB_TRY(dev_alloc(ix, &ix->d_text, ix->text_words, true));
    return KMER_B200_OK;
}

// Scheme tables, device-side descriptor, final synchronisation. ix->elems must be complete.
int finalize_index(kmer_b200_index *ix) {
    const uint32_t n_ks = (uint32_t)ix->ks.size();
    // ---- scheme tables (depend on the ks only: cached per process, a multi-k table costs ~50 ms of host time)
    {
        static std::mutex mu;
        static std::vector<SchemeHost> cache;
        std::lock_guard<std::mutex> lock(mu);
        const SchemeHost *hit = nullptr;
        for (const auto &c : cache)
            if (c.ks == ix->ks) hit = &c;
        if (!hit) {
            if (cache.size() >= 16) cache.erase(cache.begin());
            cache.emplace_back();
            cache.back().ks = ix->ks;
            build_scheme(&cache.back());
            hit = &cache.back();
        }
        ix->sum_off = hit->sum_off;
        ix->sum_elem = hit->sum_elem;
        ix->use_multi = hit->use_multi;
    }
    KB_TRY(dev_alloc(ix, &ix->d_sum_off, ix->sum_off.size(), true));
    KB_TRY(dev_alloc(ix, &ix->d_sum_elem, ix->sum_elem.size(), true));
    KB_TRY(dev_alloc(ix, &ix->d_use_multi, ix->use_multi.size(), true));
    KB_CUDA_RET(cudaMemcpyAsync(ix->d_sum_off, ix->sum_off.data(), ix->sum_off.size() * sizeof(uint32_t),
                                cudaMemcpyHostToDevice, ix->stream));
    KB_CUDA_RET(cudaMemcpyAsync(ix->d_sum_elem, ix->sum_elem.data(), ix->sum_elem.size(), cudaMemcpyHostToDevice,
                                ix->stream));
    KB_CUDA_RET(cudaMemcpyAsync(ix->d_use_multi, ix->use_multi.data(), ix->use_multi.size(), cudaMemcpyHostToDevice,
                                ix->stream));

    // ---- device-side index descriptor
    kb::DeviceIndex &D = ix->host_index;
    std::memset(&D, 0, sizeof(D));
    D.text = kb::PackedText{ix->d_text, ix->n, ix->bits, ix->sigma};
    D.owned = ix->n - ix->cfg.halo;
    D.global_base = ix->cfg.shard_begin;
    D.n_elems = n_ks;
    D.sharded = ix->sharded ? 1 : 0;
    for (uint32_t i = 0; i < n_ks; ++i) D.elem[i] = ix->elems[i].dev;
    D.scheme = kb::SchemeTables{ix->d_sum_off, ix->d_sum_elem, ix->d_use_multi};
    std::memset(D.aux_for_len, 0xFF, sizeof(D.aux_for_len));
    for (uint32_t e = 0; e < 64; ++e) {
        // saturating: only compared against 1e7 and used as slab width when < sigma^k
        const double approx = std::pow((double)ix->sigma, (double)e);
        D.pow_sigma[e] = approx > 9.0e18 ? (1ull << 63) : fast_pow(ix->sigma, (uint8_t)e);
    }
    {
        std::vector<uint32_t> order(n_ks);
        for (uint32_t i = 0; i < n_ks; ++i) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return ix->ks[a] > ix->ks[b]; });
        for (uint32_t i = 0; i < n_ks; ++i) D.elem_by_k_desc[i] = (uint8_t)order[i];
    }
    KB_TRY(dev_alloc(ix, &ix->d_index, 1, true));
    KB_CUDA_RET(cudaMemcpyAsync(ix->d_index, &D, sizeof(D), cudaMemcpyHostToDevice, ix->stream));

    // ---- finish: surface asynchronous failures and invalid ranks
    KB_CUDA_RET(cudaMemcpyAsync(ix->h_pinned, ix->d_flags, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ix->stream));
    KB_CUDA_RET(cudaStreamSynchronize(ix->stream));
    KB_CUDA_RET(cudaGetLastError());
    if (reinterpret_cast<uint32_t *>(ix->h_pinned)[0] & 1u)
        return fail(KMER_B200_ERR_INVALID_RANK, "text contains a rank >= sigma");
    return KMER_B200_OK;
}

// a record table starts[0..R] of this index's text: 0 < R < 2^32, starts[0] = 0, non-decreasing, starts[R] = n
int records_check(const kmer_b200_index *ix, const uint64_t *starts, uint64_t n_records) {
    if (n_records == 0 || n_records >= (1ull << 32)) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "n_records must be in [1, 2^32)");
    if (starts[0] != 0 || starts[n_records] != ix->n) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "starts[0] must be 0 and starts[R] = n");
    for (uint64_t r = 0; r < n_records; ++r)
        if (starts[r + 1] < starts[r]) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "record starts must not decrease");
    return KMER_B200_OK;
}

// Make ix a collection index (the table passed records_check): the device copy of the table, the boundary bitmap
// (one scatter of the record starts) and the per-m window tables of DeviceIndex.
int attach_records_impl(kmer_b200_index *ix, const uint64_t *starts, uint64_t n_records) {
    const uint64_t words = ix->n / 64 + 1;
    uint64_t *d_starts = nullptr, *d_bits = nullptr;
    const uint64_t bytes_before = ix->device_bytes;
    if (dev_alloc(ix, &d_starts, n_records + 1, true) || dev_alloc(ix, &d_bits, words, true)) {
        dev_free(ix, d_starts);
        ix->device_bytes = bytes_before;
        return KMER_B200_ERR_OUT_OF_MEMORY;
    }
    cudaMemcpyAsync(d_starts, starts, (n_records + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ix->stream);
    cudaMemsetAsync(d_bits, 0, words * sizeof(uint64_t), ix->stream);
    kb::launch_record_boundaries(d_starts, n_records, ix->n, d_bits, ix->stream);
    kb::DeviceIndex &D = ix->host_index;
    D.boundary = d_bits;
    for (uint32_t m = 0; m < 9; ++m) D.n_win[m] = 0, D.first_win[m] = UINT64_MAX;
    for (uint64_t r = 0; r < n_records; ++r) {
        const uint64_t len = starts[r + 1] - starts[r];
        for (uint32_t m = 1; m < 9 && m <= len; ++m) {
            D.n_win[m] += len - m + 1;
            D.first_win[m] = std::min(D.first_win[m], starts[r]);
        }
    }
    cudaMemcpyAsync(ix->d_index, &D, sizeof(D), cudaMemcpyHostToDevice, ix->stream);
    cudaError_t e = cudaStreamSynchronize(ix->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        cudaGetLastError();
        D.boundary = nullptr;
        dev_free(ix, d_starts);
        dev_free(ix, d_bits);
        ix->device_bytes = bytes_before;
        return fail(KMER_B200_ERR_CUDA, std::string("attach_records: ") + cudaGetErrorString(e));
    }
    ix->starts.assign(starts, starts + n_records + 1);
    ix->d_starts = d_starts;
    ix->d_boundary = d_bits;
    return KMER_B200_OK;
}

// characters -> ranks through a 256-entry table, in place (SURVEY.md 8f.3: real inputs are characters)
__global__ void __launch_bounds__(256) translate_kernel(uint8_t *__restrict__ data, uint64_t n, const uint8_t *__restrict__ lut) {
    __shared__ uint8_t s_lut[256];
    s_lut[threadIdx.x] = lut[threadIdx.x];
    __syncthreads();
    const uint64_t i0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (i0 + 16 <= n) {
        uint4 v = *reinterpret_cast<const uint4 *>(data + i0);
        uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
            w[j] = (uint32_t)s_lut[w[j] & 0xFF] | ((uint32_t)s_lut[(w[j] >> 8) & 0xFF] << 8) |
                   ((uint32_t)s_lut[(w[j] >> 16) & 0xFF] << 16) | ((uint32_t)s_lut[w[j] >> 24] << 24);
        *reinterpret_cast<uint4 *>(data + i0) = make_uint4(w[0], w[1], w[2], w[3]);
    } else {
        for (uint64_t i = i0; i < n; ++i) data[i] = s_lut[data[i]];
    }
}

int translate_on_device(kmer_b200_index *ix, uint8_t *d_data, uint64_t n, const uint8_t *lut256) {
    uint8_t *d_lut = nullptr;
    KB_TRY(dev_alloc(ix, &d_lut, 256, false));
    KB_CUDA(cudaMemcpyAsync(d_lut, lut256, 256, cudaMemcpyHostToDevice, ix->stream));
    if (n) translate_kernel<<<(unsigned)((n + 4095) / 4096), 256, 0, ix->stream>>>(d_data, n, d_lut);
    dev_free(ix, d_lut);
    KB_CUDA(cudaGetLastError());
    return 0;
}

// The two copy streams of a device (H2D / D2H next to the compute stream). Stream creation costs milliseconds: they
// are created once per device and shared (host calls on one device are short critical sections; the per-index mutex
// orders a handle's own work).
static int ensure_copy_streams(kmer_b200_index *ix) {
    if (ix->copy_in) return 0;
    static std::mutex mu;
    static cudaStream_t cached[64][3] = {};
    std::lock_guard<std::mutex> lock(mu);
    const int d = ix->device & 63;
    if (!cached[d][0]) {
        KB_CUDA(cudaStreamCreateWithFlags(&cached[d][0], cudaStreamNonBlocking));
        KB_CUDA(cudaStreamCreateWithFlags(&cached[d][1], cudaStreamNonBlocking));
        KB_CUDA(cudaStreamCreateWithFlags(&cached[d][2], cudaStreamNonBlocking));
    }
    ix->copy_in = cached[d][0];
    ix->copy_out = cached[d][1];
    ix->copy_in2 = cached[d][2];
    return 0;
}

// Streaming pack rate of this host (input bytes per second, all pool threads), measured once per process on the first
// large batch: decides how many chunks of a pinned batch travel raw (search_batch_host_chunked).
static double stream_pack_rate(const uint8_t *ranks, uint64_t n, uint32_t bits, uint32_t sigma) {
    static std::mutex mu;
    static double rate = 0;
    std::lock_guard<std::mutex> lock(mu);
    if (rate > 0) return rate;
    kb::HostPool &pool = kb::HostPool::instance();
    const unsigned T = pool.threads();
    const uint64_t ns = std::min<uint64_t>(n, 256ull << 20);
    std::vector<uint64_t> words(kb::pack_stream_words(ns, bits) + 1, 0);
    double best = 1e30;
    for (int rep = 0; rep < 2; ++rep) {  // the first pass warms the pool and the pages
        const auto t0 = std::chrono::steady_clock::now();
        pool.run(T * 4, [&](unsigned t) { kb::pack_stream_host(ranks, ns, bits, sigma, words.data(), t, T * 4); });
        best = std::min(best, std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
    }
    rate = std::max(1e8, (double)ns / best);
    return rate;
}

// The share of raw chunks that makes the host threads and the link finish together. S symbols in all, P of them packed,
// Q queries whose 16-bit lengths the host threads compute in either kind of chunk (8 bytes read + 2 written per query;
// Q = 0 for a text):  host threads (P + 10 Q) / r  =  link (S - P + P b / 8 + 2 Q) / L.  r is the streaming pack rate of
// this host measured alone, derated: inside the pipeline the packers share the memory system with two DMA streams.
static uint32_t raw_chunk_percent(double pack_rate, uint32_t bits, uint64_t n_symbols, uint64_t n_queries) {
    double link = 52e9;
    if (const char *env = std::getenv("KMER_B200_LINK_GBS")) link = std::max(1.0, std::atof(env)) * 1e9;
    const double r = 0.85 * pack_rate, S = (double)std::max<uint64_t>(n_symbols, 1), Q = (double)n_queries;
    const double P = ((S + 2.0 * Q) / link - 10.0 * Q / r) / (1.0 / r + (1.0 - bits / 8.0) / link);
    const double raw = 100.0 * (1.0 - std::max(0.0, std::min(1.0, P / S)));
    return (uint32_t)std::max(0.0, std::min(100.0, raw + 0.5));
}

// Which of n_chunks chunks travel raw for a share of raw_pct percent: spread evenly (error diffusion), the first one among
// them -- the copy engine starts on it at once while the host threads pack the next one.
static std::vector<uint8_t> raw_chunk_choice(uint32_t raw_pct, uint64_t n_chunks) {
    std::vector<uint8_t> raw(n_chunks, 0);
    uint32_t acc = raw_pct ? 99 : 0;
    for (uint64_t c = 0; c < n_chunks; ++c) {
        acc += std::min(raw_pct, 100u);
        if (acc >= 100) raw[c] = 1, acc -= 100;
    }
    return raw;
}

// A large host text (2- or 4-bit alphabets) on its way to ix->d_text: cut into chunks of whole words; the host threads
// pack chunk after chunk as a stream (kb::pack_stream_host) into a pinned ring whose slots are copied straight into
// their place in the packed text, and -- pinned input only -- the copy engine moves the other chunks as 1-byte ranks at
// the same time (pack_text_kernel turns each into words when it has arrived). Half of the PCIe time of the plain upload
// for pinned input (config 5: 54 -> 27 ms); for pageable input (std::vector storage handed over by the C++
// header) the staged copy of the driver is replaced by packing straight out of the caller's memory. On return the whole
// packed text, padding included, is ordered on ix->stream. KMER_B200_ERR_UNSUPPORTED: the caller uploads the plain way.
constexpr uint32_t kFlagPlainTextUpload = 1u << 31;  // internal bit of kmer_b200_config.reserved (create_multi sets it)

static int upload_text_stream(kmer_b200_index *ix, const uint8_t *ranks, uint64_t n) {
    constexpr int kRing = 3;
    const uint32_t bits = ix->bits, spw = 64 / bits;
    // the devices of a multi-device handle are built at the same time, each over its own PCIe link: N packers of the
    // whole text would only compete for the host cores
    if ((bits != 2 && bits != 4) || n < (64ull << 20) || (ix->cfg.reserved & kFlagPlainTextUpload) ||
        std::getenv("KMER_B200_NO_TEXT_PIPELINE"))
        return KMER_B200_ERR_UNSUPPORTED;
    KB_TRY(ensure_copy_streams(ix));
    cudaPointerAttributes attr{};
    const bool pageable = cudaPointerGetAttributes(&attr, ranks) != cudaSuccess || attr.type == cudaMemoryTypeUnregistered;
    cudaGetLastError();
    uint32_t raw_pct = 0;
    if (!pageable) {
        raw_pct = raw_chunk_percent(stream_pack_rate(ranks, n, bits, ix->sigma), bits, n, 0);
        if (const char *env = std::getenv("KMER_B200_HOST_RAW_PCT")) raw_pct = (uint32_t)std::max(0, std::min(100, std::atoi(env)));
    }
    const uint64_t chunk = 32ull << 20;  // symbols per chunk: a multiple of every spw
    const uint64_t n_chunks = (n + chunk - 1) / chunk;
    const std::vector<uint8_t> raw = raw_chunk_choice(raw_pct, n_chunks);
    const uint64_t n_raw = (uint64_t)std::count(raw.begin(), raw.end(), 1);
    kb::HostPool &pool = kb::HostPool::instance();
    const unsigned T = pool.threads();
    cudaStream_t st = ix->stream;
    uint8_t *d_raw = nullptr;  // the raw chunks, back to back
    uint64_t *h_words[kRing] = {};
    size_t cap_words[kRing] = {};
    cudaEvent_t ev_slot[kRing] = {}, ev = nullptr;
    auto cleanup = [&](int code) {
        cudaStreamSynchronize(ix->copy_in);
        if (code != 0) cudaStreamSynchronize(st);
        for (int r = 0; r < kRing; ++r) {
            if (ev_slot[r]) cudaEventDestroy(ev_slot[r]);
            pinned_put(h_words[r], cap_words[r]);
        }
        if (ev) cudaEventDestroy(ev);
        dev_free(ix, d_raw);
        return code;
    };
    for (int r = 0; r < kRing; ++r) {
        h_words[r] = (uint64_t *)pinned_get(chunk / spw * sizeof(uint64_t), &cap_words[r]);
        if (!h_words[r]) return cleanup(fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed"));
        cudaEventCreateWithFlags(&ev_slot[r], cudaEventDisableTiming);
    }
    cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (n_raw && dev_alloc(ix, &d_raw, n_raw * chunk, false)) return cleanup(KMER_B200_ERR_OUT_OF_MEMORY);
    // the padding words behind the text; the allocations (ordered on st) before the copy stream touches them
    const uint64_t n_words = kb::pack_stream_words(n, bits);
    cudaMemsetAsync(ix->d_text + n_words, 0, (ix->text_words - n_words) * sizeof(uint64_t), st);
    cudaEventRecord(ev, st);
    cudaStreamWaitEvent(ix->copy_in, ev, 0);
    ix->build_h2d = 0;
    // chunks in text order: a raw chunk costs the host nothing (one enqueue), so the copy engine always has some queued
    // while the host threads pack; the ring's slots are handed over in the same queue and come back in time
    uint64_t at = 0, used = 0;
    bool bad_rank = false;
    std::vector<uint8_t> ok(T * 4, 1);
    ix->prof.begin(K_PACK_TEXT, (double)n + (double)n * bits / 8.0, n_raw);
    for (uint64_t c = 0; c < n_chunks && !bad_rank; ++c) {
        const uint64_t s0 = c * chunk, len = std::min(chunk, n - s0);
        if (raw[c]) {
            cudaMemcpyAsync(d_raw + at, ranks + s0, len, cudaMemcpyHostToDevice, ix->copy_in);
            ix->build_h2d += len;
            cudaEventRecord(ev, ix->copy_in);
            cudaStreamWaitEvent(st, ev, 0);
            kb::launch_pack_text(d_raw + at, len, bits, ix->sigma, kb::pack_stream_words(len, bits), ix->d_text + s0 / spw, ix->d_flags, st);
            at += chunk;
            continue;
        }
        const int slot = (int)(used % kRing);
        if (used >= kRing) cudaEventSynchronize(ev_slot[slot]);
        ++used;
        pool.run(T * 4, [&](unsigned t) { ok[t] = kb::pack_stream_host(ranks + s0, len, bits, ix->sigma, h_words[slot], t, T * 4) ? 1 : 0; });
        for (uint8_t v : ok) bad_rank = bad_rank || !v;
        if (bad_rank) break;
        cudaMemcpyAsync(ix->d_text + s0 / spw, h_words[slot], kb::pack_stream_words(len, bits) * sizeof(uint64_t), cudaMemcpyHostToDevice,
                        ix->copy_in);
        ix->build_h2d += kb::pack_stream_words(len, bits) * sizeof(uint64_t);
        cudaEventRecord(ev_slot[slot], ix->copy_in);
    }
    ix->prof.end();
    if (bad_rank) return cleanup(fail(KMER_B200_ERR_INVALID_RANK, "text contains a rank >= sigma"));
    cudaEventRecord(ev, ix->copy_in);
    cudaStreamWaitEvent(st, ev, 0);
    return cleanup(0);
}

int create_impl(const uint8_t *ranks, bool ranks_on_device, uint64_t n, uint32_t sigma, const uint32_t *ks, uint32_t n_ks,
                const kmer_b200_config *cfg_in, kmer_b200_index **out, const uint8_t *lut256 = nullptr) {
    if (!out) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "out is null");
    *out = nullptr;
    if (!ranks) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "ranks is null");
    kmer_b200_index *ix = nullptr;
    int s = new_index(n, sigma, ks, n_ks, cfg_in, &ix);
    auto build = [&]() -> int {
        DeviceGuard guard(ix->device);
        // ---- text: H2D (if needed) + pack
        const uint8_t *d_ranks = ranks;
        uint8_t *d_ranks_owned = nullptr;
        int piped = KMER_B200_ERR_UNSUPPORTED;
        if (!ranks_on_device && !lut256) {  // large host texts: packed by the host threads / pipelined over PCIe
            piped = upload_text_stream(ix, ranks, n);
            if (piped != 0 && piped != KMER_B200_ERR_UNSUPPORTED) return piped;
        }
        if (piped != 0) {
            if (!ranks_on_device) {
                KB_TRY(dev_alloc(ix, &d_ranks_owned, n, false));
                KB_CUDA_RET(cudaMemcpyAsync(d_ranks_owned, ranks, n, cudaMemcpyHostToDevice, ix->stream));
                ix->build_h2d = n;
                d_ranks = d_ranks_owned;
                if (lut256) KB_TRY(translate_on_device(ix, d_ranks_owned, n, lut256));  // invalid characters map to >= sigma
            }
            ix->prof.begin(K_PACK_TEXT, (double)n + (double)n * ix->bits / 8.0);
            kb::launch_pack_text(d_ranks, n, ix->bits, sigma, ix->text_words, ix->d_text, ix->d_flags, ix->stream);
            ix->prof.end();
            if (d_ranks_owned) dev_free(ix, d_ranks_owned);
        }
        // ---- elements
        ix->elems.resize(n_ks);
        if (ix->cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS) {
            const uint32_t owner = (uint32_t)(std::max_element(ks, ks + n_ks) - ks);
            KB_TRY(build_element(ix, ks[owner], ix->elems[owner]));
            for (uint32_t i = 0; i < n_ks; ++i)
                if (i != owner) make_view(ix->elems[i], ix->elems[owner], ks[i], sigma);
            return finalize_index(ix);
        }
        for (uint32_t i = 0; i < n_ks; ++i) KB_TRY(build_element(ix, ks[i], ix->elems[i]));
        return finalize_index(ix);
    };
    if (s == 0) s = build();
    if (s != 0) {
        if (ix) kmer_b200_destroy(ix);
        return s;
    }
    *out = ix;
    return KMER_B200_OK;
}

// ---- serialization (SURVEY.md 8f.1: the thesis assumes construct-once / load-later but ships no code) --------
// File = header, packed text words, then per element: a record and the arrays keys, pos, dir. Little-endian,
// everything 8-byte aligned. Auxiliary elements are not saved (they are rebuilt on demand).
struct FileHeader {
    char magic[8];  // "KMERB200"
    uint32_t version, sigma, bits, n_ks;
    uint64_t n, text_words, shard_begin, n_total;
    uint32_t halo, mode;
    uint32_t ks[kb::kMaxElements];
};
struct FileElement {
    uint32_t k, shift, key_bits, sort_passes, key_bytes, has_keys;
    uint64_t n_kmers, dir_entries, key_space;
};
constexpr uint32_t kFileVersion = 3;  // 2: an element's sorted hashes are optional (FileElement::has_keys bit 0)
                                      // 3: has_keys bit 1 = a view of the largest k's arrays (shared positions): no arrays follow
constexpr uint32_t kFileVersionRecords = 4;  // a collection index: version 3, then R and starts[0..R] (u64) after the elements
constexpr size_t kIoChunk = 64u << 20;

// Double-buffered: h_buf holds two halves of kIoChunk bytes; the copy of chunk c + 1 runs while chunk c is written to
// (or read from) the file, so the file I/O and the PCIe copy overlap instead of alternating.
int write_device_array(kmer_b200_index *ix, FILE *f, const void *d_ptr, uint64_t bytes, void *h_buf) {
    uint8_t *half[2] = {(uint8_t *)h_buf, (uint8_t *)h_buf + kIoChunk};
    cudaEvent_t ev[2];
    cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming);
    int status = 0;
    const uint64_t n_chunks = (bytes + kIoChunk - 1) / kIoChunk;
    auto chunk_bytes = [&](uint64_t c) { return (size_t)std::min<uint64_t>(kIoChunk, bytes - c * kIoChunk); };
    if (n_chunks) {
        cudaMemcpyAsync(half[0], (const uint8_t *)d_ptr, chunk_bytes(0), cudaMemcpyDeviceToHost, ix->stream);
        cudaEventRecord(ev[0], ix->stream);
    }
    for (uint64_t c = 0; c < n_chunks && status == 0; ++c) {
        if (c + 1 < n_chunks) {
            cudaMemcpyAsync(half[(c + 1) & 1], (const uint8_t *)d_ptr + (c + 1) * kIoChunk, chunk_bytes(c + 1), cudaMemcpyDeviceToHost,
                            ix->stream);
            cudaEventRecord(ev[(c + 1) & 1], ix->stream);
        }
        if (cudaEventSynchronize(ev[c & 1]) != cudaSuccess) status = fail(KMER_B200_ERR_CUDA, "save: device to host copy failed");
        else if (fwrite(half[c & 1], 1, chunk_bytes(c), f) != chunk_bytes(c)) status = fail(KMER_B200_ERR_INVALID_ARGUMENT, "short write");
    }
    cudaStreamSynchronize(ix->stream);
    cudaEventDestroy(ev[0]);
    cudaEventDestroy(ev[1]);
    return status;
}

int read_device_array(kmer_b200_index *ix, FILE *f, void *d_ptr, uint64_t bytes, void *h_buf) {
    uint8_t *half[2] = {(uint8_t *)h_buf, (uint8_t *)h_buf + kIoChunk};
    cudaEvent_t ev[2];
    cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming);
    bool used[2] = {false, false};
    int status = 0;
    const uint64_t n_chunks = (bytes + kIoChunk - 1) / kIoChunk;
    for (uint64_t c = 0; c < n_chunks && status == 0; ++c) {
        const int h = (int)(c & 1);
        const size_t cb = (size_t)std::min<uint64_t>(kIoChunk, bytes - c * kIoChunk);
        if (used[h]) cudaEventSynchronize(ev[h]);  // the half's previous upload has left it
        if (fread(half[h], 1, cb, f) != cb) {
            status = fail(KMER_B200_ERR_INVALID_ARGUMENT, "truncated index file");
            break;
        }
        if (cudaMemcpyAsync((uint8_t *)d_ptr + c * kIoChunk, half[h], cb, cudaMemcpyHostToDevice, ix->stream) != cudaSuccess) {
            cudaGetLastError();
            status = fail(KMER_B200_ERR_CUDA, "load: host to device copy failed");
            break;
        }
        cudaEventRecord(ev[h], ix->stream);
        used[h] = true;
    }
    if (cudaStreamSynchronize(ix->stream) != cudaSuccess && status == 0) status = fail(KMER_B200_ERR_CUDA, "load: host to device copy failed");
    cudaEventDestroy(ev[0]);
    cudaEventDestroy(ev[1]);
    return status;
}

// Build auxiliary k' = m elements for the sub-k query lengths in `want` (bit m) that have none yet, memory
// permitting; returns the lengths that still have none. See DeviceIndex::aux_for_len.
uint64_t ensure_aux_elements(kmer_b200_index *ix, uint64_t want) {
    uint64_t missing = 0;
    bool changed = false;
    for (uint32_t m = 1; m < 64; ++m) {
        if (!((want >> m) & 1) || ix->host_index.aux_for_len[m] != 0xFF) continue;
        const size_t slot = ix->elems.size();
        const double key_space = std::pow((double)ix->sigma, (double)m);
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const double need = 16.0 * (double)ix->n + 4.0 * key_space + (64 << 20);  // two (key, pos) buffers + directory
        if (slot >= (size_t)kb::kMaxElements || m > ix->n || m * ix->bits > 64 || key_space > 4294967296.0 * 64 ||
            need * 1.5 > (double)free_b) {
            missing |= 1ull << m;
            continue;
        }
        HostElement he;
        if (build_element(ix, m, he, true) != 0) {
            cudaGetLastError();
            missing |= 1ull << m;
            continue;
        }
        ix->elems.push_back(he);
        ix->host_index.elem[slot] = he.dev;
        ix->host_index.aux_for_len[m] = (uint8_t)slot;
        changed = true;
    }
    if (changed)
        cudaMemcpyAsync(ix->d_index, &ix->host_index, sizeof(kb::DeviceIndex), cudaMemcpyHostToDevice, ix->stream);
    return missing;
}

enum SearchFlavor { kFlavorFull, kFlavorCountOnly };

// lanes per query, shared-memory words per query and the longest admissible query of a batch
int search_geometry(const kmer_b200_index *ix, uint64_t max_len, uint32_t mode, kb::SearchArgs *a) {
    uint64_t len_cap = std::max<uint64_t>(max_len, 1);
    // an interior shard can only complete matches of length <= halo + 1 that start in its owned range
    if (!ix->reaches_end && ix->cfg.halo + 1 < len_cap) len_cap = ix->cfg.halo + 1;
    if (mode == KMER_B200_MODE_REFERENCE_EXACT) len_cap = std::min<uint64_t>(len_cap, kb::kQuerySizeRange);
    // Lanes per query. The search is a chain of dependent gathers (offsets -> ranks -> directory -> bucket ->
    // text), so throughput = queries in flight / chain latency: short queries over an index whose buckets are
    // short (sigma^k >~ n, the usual choice of k) get one lane each; longer queries and longer candidate lists
    // get more lanes to pack / verify in parallel, up to a full warp. Measured on B200 (profiles/): config 5
    // runs at 1.1e9 queries/s with a warp per query and 7.3e9 with a lane per query.
    uint32_t group = len_cap <= 64 ? 1 : len_cap <= 128 ? 2 : len_cap <= 256 ? 4 : len_cap <= 1024 ? 8 : 32;
    if (ix->max_avg_bucket > 8.0) group = std::max(group, 8u);
    if (ix->max_avg_bucket > 64.0) group = 32;
    if (ix->cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS) group = 32;  // the kernels with view support are warp-per-query
    else if (const char *env = std::getenv("KMER_B200_GROUP")) {  // tuning override: lanes per query
        const int g = std::atoi(env);
        if (g == 1 || g == 2 || g == 4 || g == 8 || g == 32) group = (uint32_t)g;
    }
    // keep the per-CTA staging of packed queries within 48 KB (several CTAs per SM)
    while (group < 32 && (size_t)kb::search_q_words(group, ix->bits, len_cap) * 8 * (256 / group) > 48 * 1024)
        group = group == 8 ? 32 : group * 2;
    const uint32_t q_words = kb::search_q_words(group, ix->bits, len_cap);
    if ((size_t)q_words * 8 * (256 / group) > 200 * 1024)
        return fail(KMER_B200_ERR_UNSUPPORTED, "query too long for the shared-memory staging of this build");
    a->group = group;
    a->q_words = q_words;
    a->max_len = (uint32_t)len_cap;
    return 0;
}

// queries already on the device; result stays on the device
// A search in flight between its count pass and its write pass (the sharded path exchanges presence flags
// between the two).
struct PendingSearch {
    kmer_b200_index *ix = nullptr;
    kmer_b200_result *res = nullptr;
    kb::SearchArgs args{};
    uint8_t *d_unsorted = nullptr;
    uint8_t *d_defer = nullptr;
    uint64_t *d_block_sums = nullptr;
    uint32_t *d_heavy = nullptr;  // [0] = count, [1..Q] = ids of queries with long candidate lists
    uint32_t *d_hits = nullptr;   // [0] = count, [1..Q] = ids of queries with hits (what the write pass visits)
    uint32_t *d_flags = nullptr;  // u32[4] of this search: error bits, unsorted-segment count, u64 mask of sub-k lengths w/o aux
    uint64_t *h_scratch = nullptr;  // pinned, 8 words: [0] total hits, [3] gathers, [4..5] the flag words
    size_t h_scratch_cap = 0;
    bool presence_applied = false;  // deferred mode: the whole-text rule has been applied to the counts
    bool merge_checked = false;     // add_counts: the batch has no segment that the sort pass would have to visit
    // approximate search with a hit strategy (kmer_b200_approx_options; null = every hit, no distances)
    const kmer_b200_approx_options *hit_opt = nullptr;
    uint8_t *d_budget = nullptr;     // [Q]: per-query budget of the re-seeded passes (all best, strata)
    uint32_t *d_best_pos = nullptr;  // [Q]: the best pass's lowest position with d_min
    void release() {
        dev_free(ix, d_budget);
        dev_free(ix, d_best_pos);
        d_budget = nullptr;
        d_best_pos = nullptr;
        dev_free(ix, d_flags);
        d_flags = nullptr;
        pinned_put(h_scratch, h_scratch_cap);
        h_scratch = nullptr;
        dev_free(ix, d_hits);
        d_hits = nullptr;
        dev_free(ix, d_unsorted);
        dev_free(ix, d_defer);
        dev_free(ix, d_block_sums);
        dev_free(ix, d_heavy);
        d_unsorted = d_defer = nullptr;
        d_block_sums = nullptr;
        d_heavy = nullptr;
    }
};

// count pass. d_present4 != nullptr: deferred mode -- the per-part presence flags go to d_present4 and the
// whole-text presence rule is applied later by search_finish().
// queries packed before they reached the device (host threads of the host-buffer search): see SearchArgs::q_packed
struct PackedQueries {
    const uint64_t *d_words;
    const uint16_t *d_lens;
    uint32_t stride;
};

// A device result of Q queries with its offsets and status allocated, or null (the error is recorded); the caller places
// the rest and releases it with kmer_b200_result_free.
kmer_b200_result *device_result_new(kmer_b200_index *ix, uint64_t Q) {
    kmer_b200_result *res = new (std::nothrow) kmer_b200_result();
    if (!res) {
        fail(KMER_B200_ERR_OUT_OF_MEMORY, "host allocation failed");
        return nullptr;
    }
    res->index = ix;
    res->on_device = true;
    res->n_queries = Q;
    if (dev_alloc(ix, &res->offsets, Q + 1, false) || dev_alloc(ix, &res->status, Q, false)) {
        kmer_b200_result_free(res);
        return nullptr;
    }
    return res;
}

// the device arrays of a hit strategy (search_begin allocates them)
kb::ApproxHitArgs approx_hit_args(const PendingSearch *p) {
    kb::ApproxHitArgs h{};
    h.budget = p->d_budget;
    h.best_dist = p->res->best_distance;
    h.best_pos = p->d_best_pos;
    h.strata = p->hit_opt && p->hit_opt->hits == KMER_B200_HITS_STRATA ? std::min(p->hit_opt->strata, kb::kMaxMismatches) : 0;
    return h;
}

int search_begin(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint64_t max_len,
                 uint32_t mode, const void *d_present_global, uint32_t present_format, uint32_t *d_present4,
                 PendingSearch *p, const PackedQueries *packed = nullptr, int32_t max_mismatches = -1,
                 const kmer_b200_approx_options *hit_opt = nullptr) {
    using namespace kb;
    const bool collection = !ix->starts.empty();
    if (collection && max_mismatches < 0) {
        // exact search on a collection: CORRECT mode, answered by approximate search with e = 0 (the same result on a
        // plain index), whose kernels honour the record boundaries
        if (mode == KMER_B200_MODE_REFERENCE_EXACT)
            return fail(KMER_B200_ERR_INVALID_ARGUMENT, "a collection index searches in CORRECT mode only: the reference has no collections");
        if (mode != UINT32_MAX && mode != KMER_B200_MODE_CORRECT) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "unknown mode");
        if (d_present4 || d_present_global || packed)
            return fail(KMER_B200_ERR_UNSUPPORTED, "a collection index is unsharded: no cross-shard search");
        max_mismatches = 0;
    }
    const bool approx = max_mismatches >= 0;  // approximate search: the semantics of CORRECT mode, any query length
    if (approx) mode = KMER_B200_MODE_CORRECT;
    if (mode == UINT32_MAX) mode = ix->cfg.mode;
    if (mode > KMER_B200_MODE_CORRECT) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "unknown mode");
    // query ids travel as 32-bit values (heavy list, hit list, block indices of the launch)
    if (Q >= 0xFFFFFFFFull) return fail(KMER_B200_ERR_UNSUPPORTED, "more than 2^32 - 2 queries in one batch: split the batch");
    if ((ix->cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS) && (d_present4 || d_present_global))
        return fail(KMER_B200_ERR_UNSUPPORTED, "a shared-positions index is unsharded: no cross-shard presence exchange");
    cudaStream_t st = ix->stream;
    kmer_b200_result *res = device_result_new(ix, Q);
    if (!res) return KMER_B200_ERR_OUT_OF_MEMORY;
    p->ix = ix;
    p->res = res;
    auto bail = [&](int code) {
        p->release();
        kmer_b200_result_free(res);
        p->res = nullptr;
        return code;
    };
    if (dev_alloc(ix, &p->d_unsorted, Q, false) || dev_alloc(ix, &p->d_block_sums, offsets_scan_blocks(Q) + 1, false) ||
        (d_present4 && dev_alloc(ix, &p->d_defer, Q, false)) || dev_alloc(ix, &p->d_heavy, Q + 1, false) ||
        dev_alloc(ix, &p->d_hits, Q + 1, false) || dev_alloc(ix, &p->d_flags, 4, false))
        return bail(KMER_B200_ERR_OUT_OF_MEMORY);
    const bool best_pass = approx && hit_opt && hit_opt->hits != KMER_B200_HITS_ALL;
    p->hit_opt = approx ? hit_opt : nullptr;
    if (best_pass && (dev_alloc(ix, &res->best_distance, Q, false) || dev_alloc(ix, &p->d_best_pos, Q, false) ||
                      (hit_opt->hits != KMER_B200_HITS_SINGLE_BEST && dev_alloc(ix, &p->d_budget, Q, false))))
        return bail(KMER_B200_ERR_OUT_OF_MEMORY);
    p->h_scratch = (uint64_t *)pinned_get(8 * sizeof(uint64_t), &p->h_scratch_cap);
    if (!p->h_scratch) return bail(fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed"));
    cudaMemsetAsync(p->d_heavy, 0, sizeof(uint32_t), st);
    cudaMemsetAsync(p->d_hits, 0, sizeof(uint32_t), st);

    SearchArgs &a = p->args;
    a = SearchArgs{};
    if (int s = search_geometry(ix, max_len, mode, &a)) return bail(s);
    a.index = ix->d_index;
    a.q_ranks = d_q;
    a.q_offsets = d_off;
    if (packed) {
        a.q_packed = packed->d_words;
        a.q_lens16 = packed->d_lens;
        a.q_stride = packed->stride;
    }
    a.n_queries = Q;
    a.mode = mode;
    a.present_global = present_format == 0 ? (const uint64_t *)d_present_global : nullptr;
    a.present_global4 = present_format == 1 ? (const uint32_t *)d_present_global : nullptr;
    a.counts = res->offsets;
    a.status = res->status;
    a.unsorted = p->d_unsorted;
    a.positions = nullptr;
    a.present = nullptr;
    a.present4 = d_present4;
    a.defer = p->d_defer;
    a.heavy = p->d_heavy;
    a.hits = p->d_hits;
    a.bits = ix->bits;
    a.single_k = ix->ks.size() == 1;
    a.views = (ix->cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS) ? 1 : 0;
    {
        // element 0's position parts travel in the launch parameters (constant bank): the lean kernel resolves a part
        // without touching memory
        const kb::Element &E0 = ix->elems[0].dev;
        a.parts0.n = E0.n_pos_parts;
        for (int r = 0; r <= kb::kMaxPosParts; ++r) a.parts0.first[r] = E0.part_first[r];
        for (int r = 0; r < kb::kMaxPosParts; ++r) a.parts0.ptr[r] = E0.pos_part[r];
    }
    a.approx = approx ? (collection ? 2 : 1) : 0;
    a.max_mismatches = approx ? (uint32_t)max_mismatches : 0;
    a.lean_ok = !approx && a.single_k && ix->sigma == 4 && ix->elems[0].dev.shift == 0 && ix->elems[0].key_bytes == 4 && !d_present4 &&
                !d_present_global && ix->cfg.profile < 2 && !std::getenv("KMER_B200_NO_LEAN");
    a.error_flag = p->d_flags;  // per search: a second search on the handle cannot clobber a pending one's flags
    a.gather_count = ix->cfg.profile >= 2 ? ix->d_gathers : nullptr;  // profile = 2: also count gathered sectors
    if (a.gather_count) cudaMemsetAsync(ix->d_gathers, 0, sizeof(unsigned long long), st);

    cudaMemsetAsync(p->d_flags, 0, 4 * sizeof(uint32_t), st);
    if (best_pass) {
        // best pass over every query; all best and strata then count again over the queries it listed, each with its budget
        const ApproxHitArgs h = approx_hit_args(p);
        const SearchPass count = a.gather_count ? kPassCountAccount : kPassCount;
        ix->prof.begin(K_APPROX_BEST, 0);
        launch_search_approx_hits(a, h, kApproxBest, count, st);
        ix->prof.end();
        if (hit_opt->hits != KMER_B200_HITS_SINGLE_BEST) {
            cudaMemsetAsync(p->d_heavy, 0, sizeof(uint32_t), st);
            ix->prof.begin(K_SEARCH_COUNT, 0);
            launch_search_approx_hits(a, h, kApproxListed, count, st);
            ix->prof.end();
        }
    } else if (approx) {
        ix->prof.begin(K_SEARCH_COUNT, 0);
        launch_search_approx(a, a.gather_count ? kPassCountAccount : kPassCount, st);
        ix->prof.end();
    } else {
        ix->prof.begin(K_SEARCH_COUNT, 0);
        launch_search(a, d_present4 ? (a.gather_count ? kPassCountDeferredAccount : kPassCountDeferred)
                                    : (a.gather_count ? kPassCountAccount : kPassCount), st);
        ix->prof.end();
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return bail(fail(KMER_B200_ERR_CUDA, std::string("search (count pass): ") + cudaGetErrorString(e)));
    return KMER_B200_OK;
}

// deferred mode: the whole-text presence rule (kmer_index.hpp:216-227, :234 -> :119) applied to the counts of the
// count pass, once the flags of all shards are known
void apply_presence_rule(PendingSearch *p, const uint32_t *d_present4_global) {
    kmer_b200_index *ix = p->ix;
    kb::SearchArgs &a = p->args;
    ix->prof.begin(K_SEARCH_PRESENCE, 9.0 * a.n_queries);
    kb::launch_finalize_deferred(p->res->offsets, p->res->status, p->d_defer, d_present4_global, a.n_queries, ix->stream);
    ix->prof.end();
    a.present4 = nullptr;
    a.defer = nullptr;
    a.present_global4 = d_present4_global;  // the write pass applies the same rule
    p->presence_applied = true;
}

// counts[ids[i]] += add[i]; within[i] = what the count was before (the offset of that shard's list inside the
// query's merged list when shards are added in rank order)
__global__ void add_counts_kernel(uint64_t *__restrict__ counts, const int64_t *__restrict__ ids,
                                  const int64_t *__restrict__ add, uint64_t n, uint64_t n_queries,
                                  int64_t *__restrict__ within) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t q = (uint64_t)ids[i];
    if (q >= n_queries) return;
    within[i] = (int64_t)atomicAdd(reinterpret_cast<unsigned long long *>(counts + q), (unsigned long long)add[i]);
}

// [deferred: apply the whole-text presence rule] -> scan -> write pass -> segment sort
int search_finish(PendingSearch *p, const uint32_t *d_present4_global, SearchFlavor flavor, kmer_b200_result **out) {
    using namespace kb;
    kmer_b200_index *ix = p->ix;
    kmer_b200_result *res = p->res;
    cudaStream_t st = ix->stream;
    SearchArgs &a = p->args;
    const uint64_t Q = a.n_queries;
    auto bail = [&](int code) {
        p->release();
        kmer_b200_result_free(res);
        p->res = nullptr;
        return code;
    };
    if (p->d_defer && !p->presence_applied) {
        if (!d_present4_global) return bail(fail(KMER_B200_ERR_INVALID_ARGUMENT, "missing global presence flags"));
        apply_presence_rule(p, d_present4_global);
    }
    ix->prof.begin(K_OFFSETS_SCAN, 3.0 * 8 * Q, 3);
    launch_offsets_scan(res->offsets, Q, p->d_block_sums, st);
    ix->prof.end();
    // total hits + flags back to the host: the one synchronisation point of a search
    uint64_t *hs = p->h_scratch;
    cudaMemcpyAsync(&hs[0], res->offsets + Q, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(&hs[4], p->d_flags, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
    if (a.gather_count) cudaMemcpyAsync(&hs[3], ix->d_gathers, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (a.gather_count) ix->last_gathers = hs[3];
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        cudaGetLastError();
        return bail(fail(KMER_B200_ERR_CUDA, std::string("search (count pass): ") + cudaGetErrorString(e)));
    }
    const uint64_t total = hs[0];
    const uint32_t flag_words[2] = {reinterpret_cast<const uint32_t *>(&hs[4])[0], reinterpret_cast<const uint32_t *>(&hs[4])[1]};
    const uint32_t *flags = flag_words;
    const uint64_t want_aux = hs[5];  // flags[2..3]: sub-k query lengths answered by slab enumeration
    if (flags[0] & 1u) return bail(fail(KMER_B200_ERR_INVALID_RANK, "a query contains a rank >= sigma"));
    res->n_positions = total;
    // sub-k lengths seen in this batch get an auxiliary k' = m element (kept for later batches); the write pass
    // below already reads through it, so those results come out sorted and skip the segment sort
    uint64_t aux_missing = want_aux;
    if (flavor == kFlavorFull && want_aux && !(ix->cfg.reserved & KMER_B200_FLAG_NO_AUX)) aux_missing = ensure_aux_elements(ix, want_aux);
    const kmer_b200_approx_options *hit_opt = p->hit_opt;
    const uint32_t hits = hit_opt ? hit_opt->hits : (uint32_t)KMER_B200_HITS_ALL;
    const bool want_distances = hit_opt && (hit_opt->flags & KMER_B200_APPROX_DISTANCES);
    // asked-for distances are present even without a hit (an empty array, not NULL)
    if (flavor == kFlavorFull && want_distances && total == 0 && dev_alloc(ix, &res->distances, 1, false))
        return bail(KMER_B200_ERR_OUT_OF_MEMORY);
    if (flavor == kFlavorFull && total > 0 && hits == KMER_B200_HITS_SINGLE_BEST) {
        // one hit per listed query: the best pass has it already
        if (dev_alloc(ix, &res->positions, total, false) || (want_distances && dev_alloc(ix, &res->distances, total, false)))
            return bail(KMER_B200_ERR_OUT_OF_MEMORY);
        a.positions = res->positions;
        ix->prof.begin(K_APPROX_SINGLE, 0);
        launch_approx_single(a, approx_hit_args(p), res->distances, st);
        ix->prof.end();
    } else if (flavor == kFlavorFull && total > 0) {
        if (dev_alloc(ix, &res->positions, total, false) || (want_distances && dev_alloc(ix, &res->distances, total, false)))
            return bail(KMER_B200_ERR_OUT_OF_MEMORY);
        a.positions = res->positions;
        ix->prof.begin(K_SEARCH_WRITE, 0);
        if (a.approx && hits != KMER_B200_HITS_ALL)
            launch_search_approx_hits(a, approx_hit_args(p), kApproxListed, kPassWrite, st);
        else if (a.approx)
            launch_search_approx(a, kPassWrite, st);
        else
            launch_search(a, kPassWrite, st);
        ix->prof.end();
        // results written in slab order: sub-k lengths without an auxiliary element, anything seeded from a view, approximate
        // hits of several seeds or of a slab
        if (flags[1] != 0 && (aux_missing != 0 || a.views || a.approx)) {
            uint32_t *d_tmp = nullptr;
            if (dev_alloc(ix, &d_tmp, total, false)) return bail(KMER_B200_ERR_OUT_OF_MEMORY);
            const uint32_t key_bits = bit_length(ix->cfg.shard_begin + ix->n);
            ix->prof.begin(K_SEGMENT_SORT, 0);
            launch_segment_sort(res->positions, d_tmp, res->offsets, p->d_unsorted, Q, key_bits, st);
            ix->prof.end();
            dev_free(ix, d_tmp);
        }
        if (want_distances) {
            // d(p) in position order, after the sort; its gathered sectors join the count passes' under profile = 2
            ix->prof.begin(K_APPROX_DISTANCES, 0);
            launch_approx_distances(a, approx_hit_args(p), res->distances, st);
            ix->prof.end();
            if (a.gather_count) {
                cudaMemcpyAsync(&hs[3], ix->d_gathers, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
                if (cudaStreamSynchronize(st) == cudaSuccess) ix->last_gathers = hs[3];
            }
        }
    }
    res->hit_queries = p->d_hits;  // stays with the result (the sharded merge works from it)
    p->d_hits = nullptr;
    p->release();
    e = cudaGetLastError();
    if (e != cudaSuccess) {
        kmer_b200_result_free(res);
        p->res = nullptr;
        return fail(KMER_B200_ERR_CUDA, std::string("search (write pass): ") + cudaGetErrorString(e));
    }
    *out = res;
    p->res = nullptr;
    return KMER_B200_OK;
}

// queries already on the device; result stays on the device
int search_device_impl(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint64_t max_len,
                       uint32_t mode, const void *d_present_global, uint32_t present_format, SearchFlavor flavor,
                       kmer_b200_result **out, const PackedQueries *packed = nullptr, int32_t max_mismatches = -1,
                       const kmer_b200_approx_options *hit_opt = nullptr) {
    PendingSearch p;
    KB_TRY(search_begin(ix, d_q, d_off, Q, max_len, mode, d_present_global, present_format, nullptr, &p, packed, max_mismatches,
                        hit_opt));
    return search_finish(&p, nullptr, flavor, out);
}

__global__ void hashes_from_text_kernel(kb::PackedText text, uint32_t k, const uint32_t *__restrict__ pos, uint64_t n,
                                        uint64_t *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = kb::key_at(text.words, (uint64_t)pos[i], k, text.bits, text.sigma);
}

// non-empty buckets of an element: dense directory -> entries that differ from their successor; else run starts of the hashes
template <typename T>
__global__ void __launch_bounds__(256) count_steps_kernel(const T *__restrict__ v, uint64_t n, unsigned long long *out) {
    // number of i in [0, n) with v[i + 1] != v[i]
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t c = 0;
    for (; i < n; i += (uint64_t)gridDim.x * blockDim.x) c += v[i + 1] != v[i];
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, (unsigned long long)c);
}

__global__ void max_len_kernel(const uint64_t *__restrict__ off, uint64_t Q, unsigned long long *out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long m = 0;
    for (; i < Q; i += (uint64_t)gridDim.x * blockDim.x) m = max(m, (unsigned long long)(off[i + 1] - off[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// Approximate search, collections and seeding need the whole text and every position of every element on this device
// (whole or in peer parts), each bucket in ascending position order: refused (with the reason, `what` = the feature)
// for the handles where one of them lives elsewhere. views_ok: the feature also reads the views of a shared-positions
// index (the k-mer spectrum needs bucket sizes only, not their order).
int whole_index_check(const kmer_b200_index *ix, const char *what, bool views_ok = false) {
    const std::string w(what);
    if (!ix->replicas.empty()) return fail(KMER_B200_ERR_UNSUPPORTED, w + " is not available on a multi-device handle");
    if (ix->sharded || !ix->reaches_end || ix->cfg.halo != 0)
        return fail(KMER_B200_ERR_UNSUPPORTED, w + " is not available on a position-range shard");
    if (!views_ok && (ix->cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS))
        return fail(KMER_B200_ERR_UNSUPPORTED, w + " is not available on a shared-positions index");
    for (size_t e = 0; e < ix->ks.size(); ++e)
        if (ix->elems[e].dev.key_lo != 0 || ix->elems[e].dev.key_hi != UINT64_MAX)
            return fail(KMER_B200_ERR_UNSUPPORTED, w + " needs the whole key space: adopt the assembled element first");
    return KMER_B200_OK;
}

// The options of approximate search: INVALID_ARGUMENT for null options, an unknown strategy, unknown flag bits or e > 8,
// then the handle checks of whole_index_check. Every hit without distances takes the plain approximate path (null).
int approx_options_check(const kmer_b200_index *ix, const kmer_b200_approx_options *opt, const kmer_b200_approx_options **hit_opt) {
    if (!opt) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "approximate search: null options");
    if (opt->hits > KMER_B200_HITS_STRATA) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "approximate search: unknown hit strategy");
    if (opt->flags & ~(uint32_t)KMER_B200_APPROX_DISTANCES)
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "approximate search: unknown option flags");
    if (opt->max_mismatches > kb::kMaxMismatches)
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "approximate search: max_mismatches above 8");
    KB_TRY(whole_index_check(ix, "approximate search"));
    *hit_opt = (opt->hits == KMER_B200_HITS_ALL && !(opt->flags & KMER_B200_APPROX_DISTANCES)) ? nullptr : opt;
    return KMER_B200_OK;
}

// The checks of the seeding entry points: the element of k (not an auxiliary one), or INVALID_ARGUMENT; the handle checks
// of whole_index_check.
int seed_check(const kmer_b200_index *ix, uint32_t k, uint32_t *elem) {
    KB_TRY(whole_index_check(ix, "seeding"));
    for (size_t e = 0; e < ix->ks.size(); ++e)
        if (ix->ks[e] == k) {
            *elem = (uint32_t)e;
            return KMER_B200_OK;
        }
    return fail(KMER_B200_ERR_INVALID_ARGUMENT, "seeding: k is not one of the index's ks");
}

// Seeding of a batch already on the device (kmer_b200_seed_batch_device): k-mers per query -> scan -> count pass -> scan
// -> [write pass + heavy launch]. Two synchronisations: the number of k-mers (sizes kmer_counts), then the number of hits
// (sizes the positions). The caller holds the handle's lock and device.
int seed_device_impl(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint64_t max_len, uint32_t elem,
                     uint32_t max_occ, SearchFlavor flavor, kmer_b200_result **out) {
    using namespace kb;
    if (Q >= 0xFFFFFFFFull) return fail(KMER_B200_ERR_UNSUPPORTED, "more than 2^32 - 2 queries in one batch: split the batch");
    if (max_len >= (1ull << 32)) return fail(KMER_B200_ERR_UNSUPPORTED, "seeding: a query offset j is reported in 32 bits");
    cudaStream_t st = ix->stream;
    kmer_b200_result *res = device_result_new(ix, Q);
    if (!res) return KMER_B200_ERR_OUT_OF_MEMORY;
    uint64_t *d_kbase = nullptr, *d_block_sums = nullptr;
    uint32_t *d_flags = nullptr, *d_lo = nullptr;
    unsigned long long *d_n_heavy = nullptr;
    HeavySeed *d_heavy = nullptr;
    size_t hs_cap = 0;
    uint64_t *hs = nullptr;
    auto release = [&] {
        dev_free(ix, d_kbase);
        dev_free(ix, d_block_sums);
        dev_free(ix, d_flags);
        dev_free(ix, d_lo);
        dev_free(ix, d_n_heavy);
        dev_free(ix, d_heavy);
        pinned_put(hs, hs_cap);
    };
    auto bail = [&](int code) {
        release();
        kmer_b200_result_free(res);
        return code;
    };
    auto sync = [&](const char *what) -> int {
        cudaError_t e = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e == cudaSuccess) return KMER_B200_OK;
        cudaGetLastError();
        return fail(KMER_B200_ERR_CUDA, std::string(what) + cudaGetErrorString(e));
    };
    hs = (uint64_t *)pinned_get(8 * sizeof(uint64_t), &hs_cap);
    if (!hs) return bail(fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed"));
    if (dev_alloc(ix, &d_kbase, Q + 1, false) || dev_alloc(ix, &d_block_sums, offsets_scan_blocks(Q) + 1, false) ||
        dev_alloc(ix, &d_flags, 1, false) || dev_alloc(ix, &d_n_heavy, 1, false))
        return bail(KMER_B200_ERR_OUT_OF_MEMORY);
    // each query's first k-mer in the batch's k-mer order
    launch_seed_kmers_per_query(d_off, Q, ix->ks[elem], d_kbase, st);
    launch_offsets_scan(d_kbase, Q, d_block_sums, st);
    cudaMemcpyAsync(&hs[0], d_kbase + Q, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    if (int s = sync("seeding (k-mers per query): ")) return bail(s);
    res->n_kmers = Q ? hs[0] : 0;
    if (dev_alloc(ix, &res->kmer_counts, res->n_kmers, false) ||
        (flavor == kFlavorFull && dev_alloc(ix, &d_lo, res->n_kmers, false)))
        return bail(KMER_B200_ERR_OUT_OF_MEMORY);

    SeedArgs a{};
    a.index = ix->d_index;
    a.q_ranks = d_q;
    a.q_offsets = d_off;
    a.n_queries = Q;
    a.elem = elem;
    a.k = ix->ks[elem];
    a.max_occ = max_occ;
    a.coll = ix->starts.empty() ? 0 : 1;
    a.kmer_base = d_kbase;
    a.kmer_counts = res->kmer_counts;
    a.bucket_lo = d_lo;
    a.counts = res->offsets;
    a.status = res->status;
    a.n_heavy = d_n_heavy;
    a.error_flag = d_flags;
    a.gather_count = ix->cfg.profile >= 2 ? ix->d_gathers : nullptr;  // profile = 2: also count gathered sectors
    cudaMemsetAsync(d_flags, 0, sizeof(uint32_t), st);
    cudaMemsetAsync(d_n_heavy, 0, sizeof(unsigned long long), st);
    if (a.gather_count) cudaMemsetAsync(ix->d_gathers, 0, sizeof(unsigned long long), st);
    ix->prof.begin(K_SEED_COUNT, 0);
    launch_seed_count(a, st);
    ix->prof.end();
    ix->prof.begin(K_OFFSETS_SCAN, 3.0 * 8 * Q, 3);
    launch_offsets_scan(res->offsets, Q, d_block_sums, st);
    ix->prof.end();
    cudaMemcpyAsync(&hs[0], res->offsets + Q, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(&hs[1], d_n_heavy, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(&hs[2], d_flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
    if (a.gather_count) cudaMemcpyAsync(&hs[3], ix->d_gathers, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    if (int s = sync("seeding (count pass): ")) return bail(s);
    if (a.gather_count) ix->last_gathers = hs[3];
    if (hs[2] & 1u) return bail(fail(KMER_B200_ERR_INVALID_RANK, "a query contains a rank >= sigma"));
    const uint64_t total = Q ? hs[0] : 0, n_heavy = hs[1];
    res->n_positions = total;
    if (flavor == kFlavorFull && total > 0) {
        if (dev_alloc(ix, &res->positions, total, false) || dev_alloc(ix, &res->seed_offsets, total, false) ||
            (n_heavy && dev_alloc(ix, &d_heavy, n_heavy, false)))
            return bail(KMER_B200_ERR_OUT_OF_MEMORY);
        a.positions = res->positions;
        a.seed_offsets = res->seed_offsets;
        a.heavy = d_heavy;
        cudaMemsetAsync(d_n_heavy, 0, sizeof(unsigned long long), st);
        ix->prof.begin(K_SEED_WRITE, 0);
        launch_seed_write(a, st);
        ix->prof.end();
        if (a.gather_count) cudaMemcpyAsync(&hs[3], ix->d_gathers, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
        if (int s = sync("seeding (write pass): ")) return bail(s);
        if (a.gather_count) ix->last_gathers = hs[3];
    } else if (flavor == kFlavorFull && dev_alloc(ix, &res->seed_offsets, 1, false)) {
        return bail(KMER_B200_ERR_OUT_OF_MEMORY);  // a full result without hits: empty arrays, not NULL
    }
    release();
    *out = res;
    return KMER_B200_OK;
}

// stable LSD sort of (u32 key, u32 value) pairs by the low key_bits bits of the key (the build's tiled pair passes);
// *vals ends up pointing at the sorted values (the other buffers are freed)
int sort_pairs_u32(kmer_b200_index *ix, uint32_t *keys, uint32_t **vals, uint64_t n, uint32_t key_bits) {
    using namespace kb;
    cudaStream_t st = ix->stream;
    const uint32_t passes = (key_bits + kRadixBitsMax - 1) / kRadixBitsMax;
    const uint32_t bits_per_pass = (key_bits + passes - 1) / passes;
    const uint32_t mask = (1u << bits_per_pass) - 1;
    const uint32_t n_tiles = (uint32_t)((n + sort_tile_size() - 1) / sort_tile_size());
    const uint32_t n_chunks = (n_tiles + scan_chunk_tiles() - 1) / scan_chunk_tiles();
    uint32_t *k2 = nullptr, *v2 = nullptr, *tile_hist = nullptr, *chunk_sums = nullptr;
    int r = KMER_B200_OK;
    if (dev_alloc(ix, &k2, n, false) || dev_alloc(ix, &v2, n, false) || dev_alloc(ix, &tile_hist, (uint64_t)n_tiles * kRadix, false) ||
        dev_alloc(ix, &chunk_sums, (uint64_t)std::max(n_chunks, 1u) * kRadix, false)) {
        r = KMER_B200_ERR_OUT_OF_MEMORY;
    } else {
        uint32_t *kb_[2] = {keys, k2}, *vb[2] = {*vals, v2};
        int cur = 0;
        for (uint32_t p = 0; p < passes; ++p) {
            launch_hist_pairs(kb_[cur], 4, n, p * bits_per_pass, mask, tile_hist, st);
            launch_column_scan(tile_hist, n_tiles, chunk_sums, st);
            launch_scatter_pairs(kb_[cur], vb[cur], 4, n, p * bits_per_pass, mask, tile_hist, kb_[cur ^ 1], vb[cur ^ 1], st);
            cur ^= 1;
        }
        *vals = vb[cur];
        v2 = vb[cur ^ 1];
    }
    dev_free(ix, k2);
    dev_free(ix, v2);
    dev_free(ix, tile_hist);
    dev_free(ix, chunk_sums);
    return r;
}

// The checks of the record-vote entry points: those of seeding, then a record table and min_votes >= 1.
int votes_check(const kmer_b200_index *ix, uint32_t k, uint32_t min_votes, uint32_t *elem) {
    KB_TRY(seed_check(ix, k, elem));
    if (ix->starts.empty()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "record votes: the index has no records (attach_records)");
    if (min_votes == 0) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "record votes: min_votes must be >= 1");
    return KMER_B200_OK;
}

// Record votes of a batch already on the device (kmer_b200_record_votes_device): k-mers per query -> scan -> count pass ->
// [overflow path: scan of the flagged reads' events -> spill, segment sort, runs] -> scan -> write pass -> [the flagged
// reads' entries: two stable pair sorts and a scatter]. The caller holds the handle's lock and device.
int votes_device_impl(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint64_t max_len, uint32_t elem,
                      uint32_t max_occ, uint32_t min_votes, kmer_b200_result **out) {
    using namespace kb;
    (void)max_len;  // every read is walked in tiles: no length limit
    if (Q >= 0xFFFFFFFFull) return fail(KMER_B200_ERR_UNSUPPORTED, "more than 2^32 - 2 queries in one batch: split the batch");
    cudaStream_t st = ix->stream;
    kmer_b200_result *res = device_result_new(ix, Q);
    if (!res) return KMER_B200_ERR_OUT_OF_MEMORY;
    uint64_t *d_kbase = nullptr, *d_block_sums = nullptr, *d_pairs = nullptr, *d_flagged = nullptr;
    uint32_t *d_flags = nullptr, *d_counts = nullptr, *d_lo = nullptr, *d_spill = nullptr, *d_run_rec = nullptr, *d_run_votes = nullptr;
    uint32_t *d_keys = nullptr, *d_vals = nullptr, *d_c_rec = nullptr, *d_c_votes = nullptr, *d_c_read = nullptr;
    uint8_t *d_ovf = nullptr;
    unsigned long long *d_n_ovf = nullptr;
    size_t hs_cap = 0;
    uint64_t *hs = nullptr;
    auto release = [&] {
        for (uint64_t *p : {d_kbase, d_block_sums, d_pairs, d_flagged}) dev_free(ix, p);
        for (uint32_t *p : {d_flags, d_counts, d_lo, d_spill, d_run_rec, d_run_votes, d_keys, d_vals, d_c_rec, d_c_votes, d_c_read})
            dev_free(ix, p);
        dev_free(ix, d_ovf);
        dev_free(ix, d_n_ovf);
        pinned_put(hs, hs_cap);
    };
    auto bail = [&](int code) {
        release();
        kmer_b200_result_free(res);
        return code;
    };
    auto sync = [&](const char *what) -> int {
        cudaError_t e = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e == cudaSuccess) return KMER_B200_OK;
        cudaGetLastError();
        return fail(KMER_B200_ERR_CUDA, std::string(what) + cudaGetErrorString(e));
    };
    hs = (uint64_t *)pinned_get(8 * sizeof(uint64_t), &hs_cap);
    if (!hs) return bail(fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed"));
    if (dev_alloc(ix, &d_kbase, Q + 1, false) || dev_alloc(ix, &d_block_sums, offsets_scan_blocks(Q) + 1, false) ||
        dev_alloc(ix, &d_flags, 1, false) || dev_alloc(ix, &d_n_ovf, 1, false) || dev_alloc(ix, &d_pairs, Q + 1, false) ||
        dev_alloc(ix, &d_ovf, Q, false) || dev_alloc(ix, &res->kmer_hits, Q, false))
        return bail(KMER_B200_ERR_OUT_OF_MEMORY);
    launch_seed_kmers_per_query(d_off, Q, ix->ks[elem], d_kbase, st);
    launch_offsets_scan(d_kbase, Q, d_block_sums, st);
    cudaMemcpyAsync(&hs[0], d_kbase + Q, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    if (int s = sync("record votes (k-mers per query): ")) return bail(s);
    const uint64_t n_kmers = Q ? hs[0] : 0;
    if (dev_alloc(ix, &d_counts, n_kmers, false) || dev_alloc(ix, &d_lo, n_kmers, false)) return bail(KMER_B200_ERR_OUT_OF_MEMORY);

    VoteArgs a{};
    a.index = ix->d_index;
    a.q_ranks = d_q;
    a.q_offsets = d_off;
    a.n_queries = Q;
    a.elem = elem;
    a.k = ix->ks[elem];
    a.max_occ = max_occ;
    a.min_votes = min_votes;
    a.starts = ix->d_starts;
    a.n_records = ix->starts.size() - 1;
    a.record_bits = std::max<uint32_t>(1, bit_length(a.n_records - 1));
    a.kmer_base = d_kbase;
    a.kmer_counts = d_counts;
    a.bucket_lo = d_lo;
    a.counts = res->offsets;
    a.status = res->status;
    a.kmer_hits = res->kmer_hits;
    a.n_pairs = d_pairs;
    a.ovf = d_ovf;
    a.n_ovf = d_n_ovf;
    a.spill_off = d_pairs;
    a.error_flag = d_flags;
    cudaMemsetAsync(d_flags, 0, sizeof(uint32_t), st);
    cudaMemsetAsync(d_n_ovf, 0, sizeof(unsigned long long), st);
    ix->prof.begin(K_VOTES_COUNT, 0);
    launch_votes_count(a, st);
    ix->prof.end();
    cudaMemcpyAsync(&hs[1], d_n_ovf, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(&hs[2], d_flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
    if (int s = sync("record votes (count pass): ")) return bail(s);
    if (hs[2] & 1u) return bail(fail(KMER_B200_ERR_INVALID_RANK, "a query contains a rank >= sigma"));
    const uint64_t n_ovf = hs[1];
    uint64_t n_flagged = 0;  // survivors of the flagged reads
    if (n_ovf) {
        // overflow path: every flagged read's (k-mer, record) events in a segment of their own
        launch_offsets_scan(d_pairs, Q, d_block_sums, st);
        cudaMemcpyAsync(&hs[3], d_pairs + Q, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
        if (int s = sync("record votes (overflow sizes): ")) return bail(s);
        const uint64_t n_events = hs[3];
        if (dev_alloc(ix, &d_spill, n_events, false) || dev_alloc(ix, &d_run_rec, n_events, false) ||
            dev_alloc(ix, &d_run_votes, n_events, false) || dev_alloc(ix, &d_flagged, Q + 1, false))
            return bail(KMER_B200_ERR_OUT_OF_MEMORY);
        a.spill = d_spill;
        cudaMemsetAsync(d_flagged, 0, (Q + 1) * sizeof(uint64_t), st);
        ix->prof.begin(K_VOTES_OVERFLOW, 0, 3);
        launch_votes_spill(a, d_run_rec, d_run_votes, d_flagged, st);
        ix->prof.end();
        launch_offsets_scan(d_flagged, Q, d_block_sums, st);
        cudaMemcpyAsync(&hs[4], d_flagged + Q, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    }
    ix->prof.begin(K_OFFSETS_SCAN, 3.0 * 8 * Q, 3);
    launch_offsets_scan(res->offsets, Q, d_block_sums, st);
    ix->prof.end();
    cudaMemcpyAsync(&hs[0], res->offsets + Q, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    if (int s = sync("record votes (offsets): ")) return bail(s);
    const uint64_t total = Q ? hs[0] : 0;
    if (n_ovf) n_flagged = hs[4];
    if (n_flagged >= (1ull << 32)) return bail(fail(KMER_B200_ERR_UNSUPPORTED, "record votes: 2^32 or more entries of overflowed reads"));
    res->n_positions = total;
    if (dev_alloc(ix, &res->positions, total, false) || dev_alloc(ix, &res->votes, total, false))
        return bail(KMER_B200_ERR_OUT_OF_MEMORY);
    a.records = res->positions;
    a.votes = res->votes;
    ix->prof.begin(K_VOTES_WRITE, 0);
    launch_votes_write(a, st);
    ix->prof.end();
    if (n_flagged) {
        if (dev_alloc(ix, &d_keys, n_flagged, false) || dev_alloc(ix, &d_vals, n_flagged, false) || dev_alloc(ix, &d_c_rec, n_flagged, false) ||
            dev_alloc(ix, &d_c_votes, n_flagged, false) || dev_alloc(ix, &d_c_read, n_flagged, false))
            return bail(KMER_B200_ERR_OUT_OF_MEMORY);
        launch_votes_place(a, d_run_rec, d_run_votes, d_flagged, d_keys, d_vals, d_c_rec, d_c_votes, d_c_read, st);
        // stable: by votes descending, then by read; each read's entries stay in record order between equal votes
        if (int r = sort_pairs_u32(ix, d_keys, &d_vals, n_flagged, 32)) return bail(r);
        launch_votes_owner(d_vals, d_c_read, n_flagged, d_keys, st);
        if (int r = sort_pairs_u32(ix, d_keys, &d_vals, n_flagged, std::max<uint32_t>(1, bit_length(Q - 1)))) return bail(r);
        launch_votes_scatter(a, d_vals, d_c_rec, d_c_votes, d_c_read, d_flagged, n_flagged, st);
    }
    if (int s = sync("record votes (write pass): ")) return bail(s);
    release();
    *out = res;
    return KMER_B200_OK;
}

// Query lengths of a host batch: the batch and its offsets staged on the device, and the longest query. The staging is
// released with the object.
struct StagedBatch {
    kmer_b200_index *ix;
    uint8_t *d_q = nullptr;
    uint64_t *d_off = nullptr;
    unsigned long long *d_max = nullptr;
    uint64_t max_len = 0;
    explicit StagedBatch(kmer_b200_index *x) : ix(x) {}
    ~StagedBatch() {
        dev_free(ix, d_q);
        dev_free(ix, d_off);
        dev_free(ix, d_max);
    }
    // one copy each of the ranks (translated with lut256 when given) and the offsets; d_q is indexed by the caller's
    // offsets (it points q_offsets[0] symbols before the copy)
    int stage(const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q, const uint8_t *lut256) {
        cudaStream_t st = ix->stream;
        const uint64_t n_sym = q_offsets[Q] - q_offsets[0];
        KB_TRY(dev_alloc(ix, &d_q, n_sym, false));
        KB_TRY(dev_alloc(ix, &d_off, Q + 1, false));
        KB_TRY(dev_alloc(ix, &d_max, 1, false));
        KB_CUDA(cudaMemcpyAsync(d_off, q_offsets, (Q + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
        if (n_sym) KB_CUDA(cudaMemcpyAsync(d_q, q_ranks + q_offsets[0], n_sym, cudaMemcpyHostToDevice, st));
        if (lut256) KB_TRY(translate_on_device(ix, d_q, n_sym, lut256));
        KB_CUDA(cudaMemsetAsync(d_max, 0, sizeof(unsigned long long), st));
        if (Q) max_len_kernel<<<(unsigned)std::min<uint64_t>((Q + 255) / 256, (uint64_t)kb::device_sm_count() * 8), 256, 0, st>>>(d_off, Q, d_max);
        KB_CUDA(cudaMemcpyAsync(&ix->h_pinned[2], d_max, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        KB_CUDA(cudaStreamSynchronize(st));
        max_len = ix->h_pinned[2];
        return KMER_B200_OK;
    }
    const uint8_t *ranks(const uint64_t *q_offsets) const { return d_q - q_offsets[0]; }
};

// What a batch entry point asks for. Every device entry point and every single-copy host batch is one of these five kinds.
struct BatchRequest {
    enum Kind { kExact, kExactGlobal, kApprox, kSeeds, kVotes } kind = kExact;
    SearchFlavor flavor = kFlavorFull;
    uint32_t mode = UINT32_MAX;     // exact: a kmer_b200_mode, or UINT32_MAX for the index default
    const void *present = nullptr;  // exact global: the whole-text presence flags and their format
    uint32_t present_format = 0;
    const kmer_b200_approx_options *opt = nullptr;      // approximate: the caller's options
    const kmer_b200_approx_options *hit_opt = nullptr;  // approximate: the effective options (request_check)
    uint32_t k = 0, elem = 0, max_occ = 0;              // seeding, votes: k, its element (request_check) and the repeat cap
    uint32_t min_votes = 0;                             // votes: the fewest votes an entry needs
    static BatchRequest exact(uint32_t mode, SearchFlavor f) {
        BatchRequest r;
        r.mode = mode, r.flavor = f;
        return r;
    }
    static BatchRequest exact_global(uint32_t mode, const void *present, uint32_t format) {
        BatchRequest r;
        r.kind = kExactGlobal, r.mode = mode, r.present = present, r.present_format = format;
        return r;
    }
    static BatchRequest approx(const kmer_b200_approx_options *opt, SearchFlavor f) {
        BatchRequest r;
        r.kind = kApprox, r.opt = opt, r.flavor = f;
        return r;
    }
    static BatchRequest seeds(uint32_t k, uint32_t max_occ, SearchFlavor f) {
        BatchRequest r;
        r.kind = kSeeds, r.k = k, r.max_occ = max_occ, r.flavor = f;
        return r;
    }
    static BatchRequest votes(uint32_t k, uint32_t max_occ, uint32_t min_votes) {
        BatchRequest r;
        r.kind = kVotes, r.k = k, r.max_occ = max_occ, r.min_votes = min_votes;
        return r;
    }
};

// The checks of a request before the device is touched (the batch's offsets, on the host or the device, must not be
// null); fills in the effective hit options of approximate search and the element of seeding.
int request_check(const kmer_b200_index *ix, const uint64_t *offsets, BatchRequest *req, kmer_b200_result **out) {
    if (!ix || !out || !offsets) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    switch (req->kind) {
    case BatchRequest::kExactGlobal:
        if (!req->present || req->present_format > 1) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
        return KMER_B200_OK;
    case BatchRequest::kApprox: return approx_options_check(ix, req->opt, &req->hit_opt);
    case BatchRequest::kSeeds: return seed_check(ix, req->k, &req->elem);
    case BatchRequest::kVotes: return votes_check(ix, req->k, req->min_votes, &req->elem);
    default: return KMER_B200_OK;
    }
}

// A checked request over queries on the device; the result stays on the device. The caller holds the handle's lock and
// device.
int request_run(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint64_t max_len, const BatchRequest &req,
                kmer_b200_result **out) {
    switch (req.kind) {
    case BatchRequest::kApprox:
        return search_device_impl(ix, d_q, d_off, Q, max_len, KMER_B200_MODE_CORRECT, nullptr, 0, req.flavor, out, nullptr,
                                  (int32_t)req.opt->max_mismatches, req.hit_opt);
    case BatchRequest::kSeeds: return seed_device_impl(ix, d_q, d_off, Q, max_len, req.elem, req.max_occ, req.flavor, out);
    case BatchRequest::kVotes: return votes_device_impl(ix, d_q, d_off, Q, max_len, req.elem, req.max_occ, req.min_votes, out);
    default: return search_device_impl(ix, d_q, d_off, Q, max_len, req.mode, req.present, req.present_format, req.flavor, out);
    }
}

}  // namespace

extern "C" {

void kmer_b200_config_default(kmer_b200_config *cfg) {
    if (!cfg) return;
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->device = -1;
    cfg->mode = KMER_B200_MODE_REFERENCE_EXACT;
}

int kmer_b200_abi_version(void) { return KMER_B200_ABI_VERSION; }

const char *kmer_b200_last_error(void) { return g_last_error.c_str(); }

static int create_multi(const uint8_t *ranks, uint64_t n, uint32_t sigma, const uint32_t *ks, uint32_t n_ks,
                        const kmer_b200_config *cfg, kmer_b200_index **out, const uint8_t *lut256);
static int search_batch_multi(kmer_b200_index *group, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q, uint32_t mode,
                              const uint8_t *lut256, kmer_b200_result **out);
#define KB_NOT_ON_GROUP(ix)                                                                                         \
    if ((ix) && !(ix)->replicas.empty())                                                                            \
        return fail(KMER_B200_ERR_UNSUPPORTED, "device-pointer entry points are not available on a multi-device handle")
#define KB_NOT_ON_COLLECTION(ix)                                                                                    \
    if ((ix) && !(ix)->starts.empty())                                                                              \
        return fail(KMER_B200_ERR_UNSUPPORTED, "cross-shard and routed searches are not available on a collection index")

int kmer_b200_create(const uint8_t *ranks, uint64_t n, uint32_t sigma, const uint32_t *ks, uint32_t n_ks,
                     const kmer_b200_config *cfg, kmer_b200_index **out) {
    if (cfg && cfg->n_devices > 1) return create_multi(ranks, n, sigma, ks, n_ks, cfg, out, nullptr);
    return create_impl(ranks, false, n, sigma, ks, n_ks, cfg, out);
}

int kmer_b200_create_from_device(const uint8_t *d_ranks, uint64_t n, uint32_t sigma, const uint32_t *ks, uint32_t n_ks,
                                 const kmer_b200_config *cfg, kmer_b200_index **out) {
    if (cfg && cfg->n_devices > 1) return fail(KMER_B200_ERR_UNSUPPORTED, "a multi-device index is built from a host text");
    return create_impl(d_ranks, true, n, sigma, ks, n_ks, cfg, out);
}

int kmer_b200_save(kmer_b200_index *ix, const char *path) {
    if (!ix || !path) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    ix = primary(ix);  // every device of a multi-device handle holds the whole index
    if (ix->cfg.key_parts > 1) return fail(KMER_B200_ERR_UNSUPPORTED, "a key-range part is not a whole index: assemble it first");
    for (const HostElement &he : ix->elems)
        if (he.in_parts) return fail(KMER_B200_ERR_UNSUPPORTED, "the positions of this index live in several GPUs' memory: save a replicated index");
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    FILE *f = std::fopen(path, "wb");
    if (!f) return fail(KMER_B200_ERR_INVALID_ARGUMENT, std::string("cannot open ") + path);
    size_t cap = 0;
    void *h_buf = pinned_get(2 * kIoChunk, &cap);
    int s = h_buf ? 0 : fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed");
    FileHeader h{};
    std::memcpy(h.magic, "KMERB200", 8);
    h.version = ix->starts.empty() ? kFileVersion : kFileVersionRecords;
    h.sigma = ix->sigma;
    h.bits = ix->bits;
    h.n_ks = (uint32_t)ix->ks.size();
    h.n = ix->n;
    h.text_words = ix->text_words;
    h.shard_begin = ix->cfg.shard_begin;
    h.n_total = ix->cfg.n_total;
    h.halo = ix->cfg.halo;
    h.mode = ix->cfg.mode;
    for (uint32_t i = 0; i < h.n_ks; ++i) h.ks[i] = ix->ks[i];
    if (s == 0 && fwrite(&h, sizeof(h), 1, f) != 1) s = fail(KMER_B200_ERR_INVALID_ARGUMENT, "short write");
    if (s == 0) s = write_device_array(ix, f, ix->d_text, ix->text_words * 8, h_buf);
    for (uint32_t i = 0; s == 0 && i < h.n_ks; ++i) {
        const HostElement &he = ix->elems[i];
        FileElement fe{he.dev.k, he.dev.shift, he.key_bits, he.sort_passes, he.key_bytes, he.d_keys ? 1u : 0u, he.dev.n_kmers,
                       he.dev.dir_entries, he.dev.key_space};
        if (he.view) fe = FileElement{he.dev.k, 0, he.key_bits, 0, he.key_bytes, 2u, 0, 0, 0};
        if (fwrite(&fe, sizeof(fe), 1, f) != 1) s = fail(KMER_B200_ERR_INVALID_ARGUMENT, "short write");
        if (he.view) continue;
        if (s == 0 && he.d_keys) s = write_device_array(ix, f, he.d_keys, he.dev.n_kmers * he.key_bytes, h_buf);
        if (s == 0) s = write_device_array(ix, f, he.d_pos, he.dev.n_kmers * 4, h_buf);
        if (s == 0) s = write_device_array(ix, f, he.d_dir, he.dev.dir_entries * 4, h_buf);
    }
    if (s == 0 && !ix->starts.empty()) {
        const uint64_t n_records = ix->starts.size() - 1;
        if (fwrite(&n_records, sizeof(n_records), 1, f) != 1 || fwrite(ix->starts.data(), sizeof(uint64_t), n_records + 1, f) != n_records + 1)
            s = fail(KMER_B200_ERR_INVALID_ARGUMENT, "short write");
    }
    pinned_put(h_buf, cap);
    if (std::fclose(f) != 0 && s == 0) s = fail(KMER_B200_ERR_INVALID_ARGUMENT, "close failed");
    return s;
}

int kmer_b200_load(const char *path, const kmer_b200_config *cfg_in, kmer_b200_index **out) {
    if (!path || !out) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    FILE *f = std::fopen(path, "rb");
    if (!f) return fail(KMER_B200_ERR_INVALID_ARGUMENT, std::string("cannot open ") + path);
    FileHeader h{};
    if (fread(&h, sizeof(h), 1, f) != 1 || std::memcmp(h.magic, "KMERB200", 8) != 0 || h.version < 2 || h.version > kFileVersionRecords ||
        h.n_ks == 0 || h.n_ks > (uint32_t)kb::kMaxElements) {
        std::fclose(f);
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "not a kmer_b200 index file (or an unknown version)");
    }
    kmer_b200_config cfg;
    if (cfg_in)
        cfg = *cfg_in;
    else
        kmer_b200_config_default(&cfg);
    cfg.shard_begin = h.shard_begin;  // the geometry is a property of the stored index
    cfg.n_total = h.n_total;
    cfg.halo = h.halo;
    if (!cfg_in) cfg.mode = h.mode;
    kmer_b200_index *ix = nullptr;
    int s = new_index(h.n, h.sigma, h.ks, h.n_ks, &cfg, &ix);
    auto load = [&]() -> int {
        DeviceGuard guard(ix->device);
        if (ix->bits != h.bits || ix->text_words != h.text_words)
            return fail(KMER_B200_ERR_INVALID_ARGUMENT, "index file does not match this build's text packing");
        size_t cap = 0;
        void *h_buf = pinned_get(2 * kIoChunk, &cap);
        if (!h_buf) return fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed");
        int r = read_device_array(ix, f, ix->d_text, ix->text_words * 8, h_buf);
        ix->elems.resize(h.n_ks);
        const uint32_t owner = (uint32_t)(std::max_element(h.ks, h.ks + h.n_ks) - h.ks);
        uint32_t n_views = 0;
        for (uint32_t i = 0; r == 0 && i < h.n_ks; ++i) {
            HostElement &he = ix->elems[i];
            FileElement fe{};
            if (fread(&fe, sizeof(fe), 1, f) == 1 && fe.k == h.ks[i] && fe.has_keys == 2 && h.version >= 3 && i != owner) {
                he.view = true;  // filled in from the owner below
                ++n_views;
                continue;
            }
            if (fe.k != h.ks[i] || (fe.key_bytes != 4 && fe.key_bytes != 8) ||
                fe.n_kmers != h.n - fe.k + 1) {
                r = fail(KMER_B200_ERR_INVALID_ARGUMENT, "corrupt element record");
                break;
            }
            {
                // everything that drives device indexing is recomputed from (sigma, k, shift) and must agree with the file
                const uint64_t key_space = fast_pow(h.sigma, (uint8_t)fe.k);
                const uint32_t key_bits = std::max<uint32_t>(1, bit_length(key_space - 1));
                if (fe.key_space != key_space || fe.key_bits != key_bits || fe.key_bytes != (key_bits > 32 ? 8u : 4u) ||
                    fe.shift > key_bits || key_bits > 32 + fe.shift || fe.dir_entries != ((key_space - 1) >> fe.shift) + 2 ||
                    fe.sort_passes == 0 || fe.sort_passes > 64 || fe.has_keys > 1 || (fe.shift != 0 && !fe.has_keys)) {
                    r = fail(KMER_B200_ERR_INVALID_ARGUMENT, "element record inconsistent with sigma / k / shift");
                    break;
                }
            }
            he.key_bits = fe.key_bits;
            he.sort_passes = fe.sort_passes;
            he.key_bytes = fe.key_bytes;
            uint8_t *keys = nullptr;
            if (fe.has_keys && (r = dev_alloc(ix, &keys, fe.n_kmers * fe.key_bytes, true)) != 0) break;
            he.d_keys = keys;
            if ((r = dev_alloc(ix, &he.d_pos, fe.n_kmers, true)) != 0) break;
            if ((r = dev_alloc(ix, &he.d_dir, fe.dir_entries, true)) != 0) break;
            if (fe.has_keys && (r = read_device_array(ix, f, he.d_keys, fe.n_kmers * fe.key_bytes, h_buf)) != 0) break;
            if ((r = read_device_array(ix, f, he.d_pos, fe.n_kmers * 4, h_buf)) != 0) break;
            if ((r = read_device_array(ix, f, he.d_dir, fe.dir_entries * 4, h_buf)) != 0) break;
            {
                uint32_t ends[2] = {1, 0};  // dir[0] must be 0 and the last entry n_kmers (a CSR offset array)
                cudaMemcpyAsync(&ends[0], he.d_dir, 4, cudaMemcpyDeviceToHost, ix->stream);
                cudaMemcpyAsync(&ends[1], he.d_dir + fe.dir_entries - 1, 4, cudaMemcpyDeviceToHost, ix->stream);
                if (cudaStreamSynchronize(ix->stream) != cudaSuccess || ends[0] != 0 || ends[1] != (uint32_t)fe.n_kmers) {
                    r = fail(KMER_B200_ERR_INVALID_ARGUMENT, "corrupt directory in index file");
                    break;
                }
            }
            he.dev = kb::Element{fe.k, fe.shift, fe.n_kmers, fe.dir_entries, fe.key_space, he.d_dir, he.d_keys, he.d_pos,
                                 fe.key_bytes, fe.k, 0, UINT64_MAX, 1};
            he.bytes = fe.n_kmers * (4 + (fe.has_keys ? fe.key_bytes : 0)) + fe.dir_entries * 4;
            ix->max_avg_bucket = std::max(ix->max_avg_bucket,
                                          (double)fe.n_kmers / (double)std::min<uint64_t>(fe.key_space, fe.n_kmers));
        }
        pinned_put(h_buf, cap);
        if (r == 0 && n_views) {
            if (n_views + 1 != h.n_ks || ix->elems[owner].view) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "corrupt element record");
            for (uint32_t i = 0; i < h.n_ks; ++i)
                if (i != owner) make_view(ix->elems[i], ix->elems[owner], h.ks[i], h.sigma);
            ix->cfg.reserved |= KMER_B200_FLAG_SHARED_POSITIONS | KMER_B200_FLAG_NO_AUX;
        } else {
            ix->cfg.reserved &= ~(uint32_t)KMER_B200_FLAG_SHARED_POSITIONS;  // what the file holds decides
        }
        std::vector<uint64_t> rec;  // version 4: the record table of a collection index
        if (r == 0 && h.version >= kFileVersionRecords) {
            uint64_t n_records = 0;
            if (fread(&n_records, sizeof(n_records), 1, f) != 1 || n_records == 0 || n_records >= (1ull << 32))
                return fail(KMER_B200_ERR_INVALID_ARGUMENT, "corrupt record table in index file");
            rec.resize(n_records + 1);
            if (fread(rec.data(), sizeof(uint64_t), n_records + 1, f) != n_records + 1)
                return fail(KMER_B200_ERR_INVALID_ARGUMENT, "truncated index file");
            if ((r = records_check(ix, rec.data(), n_records)) != 0) return r;
        }
        if (r == 0) r = finalize_index(ix);
        if (r == 0 && !rec.empty()) r = whole_index_check(ix, "a collection index");
        if (r == 0 && !rec.empty()) r = attach_records_impl(ix, rec.data(), rec.size() - 1);
        return r;
    };
    if (s == 0) s = load();
    std::fclose(f);
    if (s != 0) {
        if (ix) kmer_b200_destroy(ix);
        return s;
    }
    *out = ix;
    return KMER_B200_OK;
}

void kmer_b200_destroy(kmer_b200_index *ix) {
    if (!ix) return;
    if (!ix->replicas.empty()) {
        for (kmer_b200_index *r : ix->replicas) kmer_b200_destroy(r);
        delete ix;
        return;
    }
    DeviceGuard guard(ix->device);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    ix->prof.resolve();
    for (auto &he : ix->elems) {
        if (he.adopted != 1) {
            dev_free(ix, he.d_dir);
            dev_free(ix, he.d_pos);
        }
        dev_free(ix, (uint8_t *)he.d_keys);
    }
    dev_free(ix, ix->d_text);
    dev_free(ix, ix->d_starts);
    dev_free(ix, ix->d_boundary);
    dev_free(ix, ix->d_sum_off);
    dev_free(ix, ix->d_sum_elem);
    dev_free(ix, ix->d_use_multi);
    dev_free(ix, ix->d_index);
    dev_free(ix, ix->d_flags);
    dev_free(ix, ix->d_gathers);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    pinned_put(ix->h_pinned, ix->h_pinned_cap);
    for (auto e : ix->prof.pool) cudaEventDestroy(e);
    ix->prof.pool.clear();
    if (ix->own_stream && ix->stream) cudaStreamDestroy(ix->stream);
    cudaGetLastError();
    delete ix;
}

// The device entry points: the request's checks, then the device and the handle's lock, once for all of them. The exact
// forms refuse multi-device handles first, the global-presence form collection indexes too; approximate search and
// seeding (record votes too) refuse those handles in their own checks.
static int device_entry(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint64_t max_len, BatchRequest req,
                        kmer_b200_result **out) {
    if (req.kind == BatchRequest::kExact || req.kind == BatchRequest::kExactGlobal) { KB_NOT_ON_GROUP(ix); }
    if (req.kind == BatchRequest::kExactGlobal) { KB_NOT_ON_COLLECTION(ix); }
    KB_TRY(request_check(ix, d_off, &req, out));
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    return request_run(ix, d_q, d_off, Q, max_len, req, out);
}

int kmer_b200_search_batch_device(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q,
                                  uint64_t max_len, uint32_t mode, kmer_b200_result **out) {
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::exact(mode, kFlavorFull), out);
}

int kmer_b200_count_batch_device(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q,
                                 uint64_t max_len, uint32_t mode, kmer_b200_result **out) {
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::exact(mode, kFlavorCountOnly), out);
}

int kmer_b200_search_approx_batch_device(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q,
                                         uint64_t max_len, uint32_t max_mismatches, kmer_b200_result **out) {
    const kmer_b200_approx_options opt{max_mismatches, KMER_B200_HITS_ALL, 0, 0};
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::approx(&opt, kFlavorFull), out);
}

int kmer_b200_count_approx_batch_device(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q,
                                        uint64_t max_len, uint32_t max_mismatches, kmer_b200_result **out) {
    const kmer_b200_approx_options opt{max_mismatches, KMER_B200_HITS_ALL, 0, 0};
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::approx(&opt, kFlavorCountOnly), out);
}

int kmer_b200_search_approx_batch_device_ex(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q,
                                            uint64_t max_len, const kmer_b200_approx_options *opt, kmer_b200_result **out) {
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::approx(opt, kFlavorFull), out);
}

int kmer_b200_count_approx_batch_device_ex(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q,
                                           uint64_t max_len, const kmer_b200_approx_options *opt, kmer_b200_result **out) {
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::approx(opt, kFlavorCountOnly), out);
}

int kmer_b200_search_batch_device_global(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q,
                                         uint64_t max_len, uint32_t mode, const void *d_present_global,
                                         uint32_t present_format, kmer_b200_result **out) {
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::exact_global(mode, d_present_global, present_format), out);
}

int kmer_b200_seed_batch_device(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint64_t max_len,
                                uint32_t k, uint32_t max_occ, kmer_b200_result **out) {
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::seeds(k, max_occ, kFlavorFull), out);
}

int kmer_b200_count_seeds_batch_device(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint64_t max_len,
                                       uint32_t k, uint32_t max_occ, kmer_b200_result **out) {
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::seeds(k, max_occ, kFlavorCountOnly), out);
}

int kmer_b200_record_votes_device(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint64_t max_len,
                                  uint32_t k, uint32_t max_occ, uint32_t min_votes, kmer_b200_result **out) {
    return device_entry(ix, d_q, d_off, Q, max_len, BatchRequest::votes(k, max_occ, min_votes), out);
}

struct kmer_b200_pending {
    PendingSearch p;
};

int kmer_b200_search_sharded_begin(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q,
                                   uint64_t max_len, uint32_t mode, uint32_t *d_present4, kmer_b200_pending **out) {
    KB_NOT_ON_GROUP(ix);
    KB_NOT_ON_COLLECTION(ix);
    if (!ix || !out || !d_off || !d_present4) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    kmer_b200_pending *h = new (std::nothrow) kmer_b200_pending();
    if (!h) return fail(KMER_B200_ERR_OUT_OF_MEMORY, "host allocation failed");
    int s = search_begin(ix, d_q, d_off, Q, max_len, mode, nullptr, 0, d_present4, &h->p);
    if (s != 0) {
        delete h;
        return s;
    }
    *out = h;
    return KMER_B200_OK;
}

int kmer_b200_search_sharded_finish(kmer_b200_pending *h, const uint32_t *d_present4_global, kmer_b200_result **out) {
    if (!h || !out || !d_present4_global) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    kmer_b200_index *ix = h->p.ix;
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    int s = search_finish(&h->p, d_present4_global, kFlavorFull, out);
    delete h;
    return s;
}

void kmer_b200_search_sharded_abort(kmer_b200_pending *h) {
    if (!h) return;
    kmer_b200_index *ix = h->p.ix;
    {
        DeviceGuard guard(ix->device);
        std::lock_guard<std::mutex> lock(ix->mu);
        h->p.release();
    }
    kmer_b200_result_free(h->p.res);  // takes the device guard itself
    delete h;
}

int kmer_b200_search_sharded_peek(kmer_b200_pending *h, const uint32_t *d_present4_global, const uint64_t **d_counts_out,
                                  const uint32_t **d_hit_queries_out) {
    if (!h || !d_present4_global || !d_counts_out || !d_hit_queries_out)
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    kmer_b200_index *ix = h->p.ix;
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    if (h->p.d_defer && !h->p.presence_applied) apply_presence_rule(&h->p, d_present4_global);
    *d_counts_out = h->p.res->offsets;  // per-query counts until finish turns them into offsets
    *d_hit_queries_out = h->p.d_hits;
    return KMER_B200_OK;
}

int kmer_b200_search_sharded_add_counts(kmer_b200_pending *h, const uint32_t *d_present4_global, const int64_t *d_ids,
                                        const int64_t *d_counts, uint64_t n, int64_t *d_within_out) {
    if (!h || !d_present4_global || (n && (!d_ids || !d_counts || !d_within_out)))
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    kmer_b200_index *ix = h->p.ix;
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    if (!h->p.merge_checked) {
        // results that still need the segment sort (sub-k slabs without an auxiliary element) are sorted over
        // [offsets[q], offsets[q + 1]), which must then hold this shard's hits only: the caller merges afterwards
        uint32_t n_unsorted = 0;
        cudaError_t e = cudaMemcpyAsync(&n_unsorted, h->p.d_flags + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, ix->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ix->stream);
        if (e != cudaSuccess) return fail(KMER_B200_ERR_CUDA, std::string("add_counts: ") + cudaGetErrorString(e));
        if (n_unsorted != 0)
            return fail(KMER_B200_ERR_UNSUPPORTED, "this batch needs the segment sort: merge after kmer_b200_search_sharded_finish");
        h->p.merge_checked = true;
    }
    if (h->p.d_defer && !h->p.presence_applied) apply_presence_rule(&h->p, d_present4_global);
    if (n)
        add_counts_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ix->stream>>>(h->p.res->offsets, d_ids, d_counts, n,
                                                                               h->p.args.n_queries, d_within_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(KMER_B200_ERR_CUDA, std::string("add_counts: ") + cudaGetErrorString(e));
    return KMER_B200_OK;
}

int kmer_b200_presence_batch_device(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q,
                                    uint64_t max_len, uint32_t mode, void *d_present, uint32_t present_format) {
    KB_NOT_ON_GROUP(ix);
    KB_NOT_ON_COLLECTION(ix);
    using namespace kb;
    if (!ix || !d_off || !d_present || present_format > 1) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    if (ix->cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS)
        return fail(KMER_B200_ERR_UNSUPPORTED, "a shared-positions index is unsharded: no cross-shard presence exchange");
    if (mode == UINT32_MAX) mode = ix->cfg.mode;
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    SearchArgs a{};
    KB_TRY(search_geometry(ix, max_len, mode, &a));
    a.index = ix->d_index;
    a.q_ranks = d_q;
    a.q_offsets = d_off;
    a.n_queries = Q;
    a.mode = mode;
    a.present = present_format == 0 ? (uint64_t *)d_present : nullptr;
    a.present4 = present_format == 1 ? (uint32_t *)d_present : nullptr;
    a.bits = ix->bits;
    a.single_k = ix->ks.size() == 1;
    a.error_flag = ix->d_flags;
    ix->prof.begin(K_SEARCH_PRESENCE, 0);
    launch_search(a, kPassPresence, ix->stream);
    ix->prof.end();
    KB_CUDA(cudaGetLastError());
    return KMER_B200_OK;
}

__global__ void __launch_bounds__(256) add_base32_kernel(const uint32_t *__restrict__ src, uint64_t n, uint32_t base,
                                                         uint32_t *__restrict__ dst) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i] + base;
}

__global__ void __launch_bounds__(256) add_base_kernel(uint64_t *__restrict__ v, uint64_t n, uint64_t base) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] += base;
}

__global__ void __launch_bounds__(256) widen_lens_kernel(const uint16_t *__restrict__ lens, uint64_t n, uint64_t *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = lens[i];
}

// The host copy of a search result of Q queries: offsets and status pinned; null when an allocation failed. The positions
// are placed by host_result_positions once their number is known.
static kmer_b200_result *host_result_new(kmer_b200_index *ix, uint64_t Q) {
    kmer_b200_result *res = new (std::nothrow) kmer_b200_result();
    if (!res) return nullptr;
    res->index = ix;
    res->on_device = false;
    res->n_queries = Q;
    res->offsets = (uint64_t *)pinned_get((Q + 1) * sizeof(uint64_t), &res->cap_offsets);
    res->status = (uint8_t *)pinned_get(Q, &res->cap_status);
    if (!res->offsets || !res->status) {
        kmer_b200_result_free(res);
        return nullptr;
    }
    return res;
}

// Room for n_positions positions: pinned up to 8 GiB, pageable beyond (pinning tens of gigabytes is slow and can starve
// the host). False when the allocation failed.
static bool host_result_positions(kmer_b200_result *res, uint64_t n_positions) {
    res->n_positions = n_positions;
    const size_t pos_bytes = n_positions * sizeof(uint32_t);
    if (pos_bytes > (8ull << 30)) {
        res->positions = (uint32_t *)std::malloc(pos_bytes);
        res->positions_pageable = true;
        res->cap_positions = pos_bytes;
    } else {
        res->positions = (uint32_t *)pinned_get(pos_bytes, &res->cap_positions);
    }
    return res->positions != nullptr;
}

// A stream of packed symbols (query boundaries ignored: kb::pack_stream_host) -> the fixed-stride per-query words the
// search kernels take (SearchArgs::q_packed). One thread per output word: a funnel shift of two stream words, the
// symbols behind the query's end zeroed. `off` = symbol offsets of the queries inside the stream.
__global__ void __launch_bounds__(256) align_stream_kernel(const uint64_t *__restrict__ stream, const uint64_t *__restrict__ off,
                                                           const uint16_t *__restrict__ lens, uint64_t n_queries, uint32_t stride,
                                                           uint32_t bits, uint64_t *__restrict__ out) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_queries * stride) return;
    const uint64_t q = idx / stride;
    const uint32_t w = (uint32_t)(idx - q * stride);
    const uint32_t spw = 64 / bits;
    const uint32_t m = lens[q];
    uint64_t v = 0;
    if (w * spw < m) {
        const uint64_t bit = (off[q] + (uint64_t)w * spw) * bits;
        const uint64_t j = bit >> 6;
        const uint32_t r = (uint32_t)(bit & 63);
        v = stream[j] << r;
        if (r) v |= stream[j + 1] >> (64 - r);  // the stream carries one word of padding
        const uint32_t n_valid = min(spw, m - w * spw);
        if (n_valid < spw) v &= ~0ull << (64 - bits * n_valid);
    }
    out[idx] = v;
}

// Large host batches, in chunks of queries: the H2D copy of later chunks, the search of chunk c and the D2H copy of
// earlier chunks' offsets and status run concurrently. Per-query packing on the host cores costs more than the PCIe bytes
// it saves (16 cores pack ~30 GB/s of variable-length queries, the link moves 55 GB/s). What the host cores do fast is a
// pure streaming pack of the concatenated ranks, query boundaries ignored (kb::pack_stream_host: 128 ranks -> 32 bytes in
// ten AVX2 instructions, bound by what a core streams from DRAM: ~100 GB/s on 16 cores); cutting that stream into
// per-query words is a ~1 ms kernel on the device (align_stream_kernel). The batch is cut into chunks of queries of two
// kinds that keep BOTH resources busy:
//   * packed chunks: 16-bit lengths + streaming pack by the pool, then (bits / 8) of the bytes over PCIe;
//   * raw chunks (`raw_pct` percent of the chunks): the copy engine moves the caller's 1-byte ranks as they are -- no host
//     work beyond the lengths. A raw chunk with a query of 65 536 symbols or more sends its offsets as they are instead.
// A producer thread walks the chunks in order and never waits for the device except for a free slot of the pinned ring:
// raw chunks are queued on one H2D stream, packed chunks on another, so neither kind waits behind the other. The calling
// thread searches the chunks in order as they arrive (device buffers are allocated up front, so the producer makes no
// stream-ordered allocation); offsets and status of finished chunks leave on the D2H stream. Position lists stay on the
// device until the last chunk is done (their total size is only known then) and are copied out in one sweep. Results
// are identical to the single-copy path's (tests/test_gpu_full_size.py). KMER_B200_ERR_UNSUPPORTED: a packed chunk holds
// a query longer than 16 words or 65 535 symbols, or no producer thread could be started.
static int search_batch_host_chunked(kmer_b200_index *ix, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q,
                                     uint32_t mode, uint32_t raw_pct, kmer_b200_result **out) {
    constexpr int kChunks = 24, kRing = 4;
    // KMER_B200_HOST_TRACE=1: where the time went (ms), printed to stderr at the end of the call
    const bool trace = std::getenv("KMER_B200_HOST_TRACE") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto since = [](std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
    const auto t_call = now();
    double t_wait_chunk = 0, t_search = 0;                       // calling thread
    double t_slot = 0, t_pool = 0, t_enqueue = 0, t_producer = 0;  // producer thread
    cudaStream_t st = ix->stream;
    KB_TRY(ensure_copy_streams(ix));
    kb::HostPool &pool = kb::HostPool::instance();
    const unsigned T = pool.threads();
    const uint32_t bits = ix->bits, spw = 64 / bits, sigma = ix->sigma;
    const uint64_t per = (Q + kChunks - 1) / kChunks;
    uint64_t c0[kChunks + 1];
    for (int c = 0; c <= kChunks; ++c) c0[c] = std::min<uint64_t>((uint64_t)c * per, Q);
    const std::vector<uint8_t> raw = raw_chunk_choice(raw_pct, kChunks);

    const uint64_t max_stride = 16;
    uint16_t *h_lens = nullptr;
    size_t cap_lens = 0;
    uint64_t *h_words[kRing] = {};
    size_t cap_words[kRing] = {};
    void *d_in[kChunks] = {};        // raw chunk: its ranks; packed chunk: its packed stream (+ one word of padding)
    uint64_t *d_words[kChunks] = {}; // packed chunk: per-query words after the alignment
    uint16_t *d_lens[kChunks] = {};
    uint64_t *d_off[kChunks] = {};   // chunk-relative symbol offsets, rebuilt on the device
    bool lens16[kChunks] = {};       // the chunk sent 16-bit lengths (else its offsets as they are)
    uint64_t *d_scan = nullptr;
    uint32_t stride[kChunks] = {};
    uint64_t max_len[kChunks] = {}, n_sym_c[kChunks] = {}, n_stream_words[kChunks] = {};
    kmer_b200_result *chunk_res[kChunks] = {};
    cudaEvent_t ev_in[kChunks] = {}, ev_done[kChunks] = {}, ev_slot[kRing] = {};
    kmer_b200_result *res = nullptr;
    // producer -> calling thread
    std::mutex mu;
    std::condition_variable cv;
    int produced = 0;                // chunks [0, produced) are queued on a copy stream
    bool producer_failed = false;    // unsupported / bad rank / allocation: see the flags
    std::atomic<bool> stop{false};
    bool unsupported = false, bad_rank = false;
    uint64_t h2d = 0;
    std::thread producer;
    auto cleanup = [&](int code) {
        stop.store(true);
        if (producer.joinable()) producer.join();
        cudaStreamSynchronize(ix->copy_in);
        cudaStreamSynchronize(ix->copy_in2);
        cudaStreamSynchronize(ix->copy_out);
        cudaStreamSynchronize(st);
        for (int c = 0; c < kChunks; ++c) {
            if (chunk_res[c]) kmer_b200_result_free(chunk_res[c]);
            if (ev_in[c]) cudaEventDestroy(ev_in[c]);
            if (ev_done[c]) cudaEventDestroy(ev_done[c]);
            dev_free(ix, (uint8_t *)d_in[c]);
            dev_free(ix, d_words[c]);
            dev_free(ix, d_lens[c]);
            dev_free(ix, d_off[c]);
        }
        dev_free(ix, d_scan);
        for (int r = 0; r < kRing; ++r) {
            if (ev_slot[r]) cudaEventDestroy(ev_slot[r]);
            pinned_put(h_words[r], cap_words[r]);
        }
        pinned_put(h_lens, cap_lens);
        if (code != 0 && res) kmer_b200_result_free(res);
        return code;
    };
    h_lens = (uint16_t *)pinned_get(std::max<uint64_t>(Q, 1) * sizeof(uint16_t), &cap_lens);
    if (!h_lens) return cleanup(fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed"));
    uint64_t ring_words = 1;
    for (int c = 0; c < kChunks; ++c) {
        n_sym_c[c] = q_offsets[c0[c + 1]] - q_offsets[c0[c]];
        n_stream_words[c] = kb::pack_stream_words(n_sym_c[c], bits);
        if (!raw[c]) ring_words = std::max(ring_words, n_stream_words[c] + 1);
        cudaEventCreateWithFlags(&ev_in[c], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&ev_done[c], cudaEventDisableTiming);
    }
    for (int r = 0; r < kRing; ++r) {
        h_words[r] = (uint64_t *)pinned_get(ring_words * sizeof(uint64_t), &cap_words[r]);
        if (!h_words[r]) return cleanup(fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed"));
        cudaEventCreateWithFlags(&ev_slot[r], cudaEventDisableTiming);
    }
    // every device buffer the copy streams write, allocated now (stream-ordered on `st`) and fenced once
    if (dev_alloc(ix, &d_scan, kb::offsets_scan_blocks(per) + 1, false)) return cleanup(KMER_B200_ERR_OUT_OF_MEMORY);
    for (int c = 0; c < kChunks; ++c) {
        const uint64_t Qc = c0[c + 1] - c0[c];
        if (Qc == 0) continue;
        uint8_t *bytes = nullptr;
        if (dev_alloc(ix, &d_lens[c], Qc, false) || dev_alloc(ix, &d_off[c], Qc + 1, false) ||
            dev_alloc(ix, &bytes, raw[c] ? n_sym_c[c] : (n_stream_words[c] + 1) * sizeof(uint64_t), false))
            return cleanup(KMER_B200_ERR_OUT_OF_MEMORY);
        d_in[c] = bytes;
    }
    {
        cudaEvent_t ev0;  // no copy stream runs ahead of the allocations or of work already queued on `st`
        cudaEventCreateWithFlags(&ev0, cudaEventDisableTiming);
        cudaEventRecord(ev0, st);
        cudaStreamWaitEvent(ix->copy_in, ev0, 0);
        cudaStreamWaitEvent(ix->copy_in2, ev0, 0);
        cudaStreamWaitEvent(ix->copy_out, ev0, 0);
        cudaEventDestroy(ev0);
    }
    res = host_result_new(ix, Q);
    if (!res) return cleanup(fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed"));

    const int device = ix->device;
    auto produce = [&] {
        cudaSetDevice(device);
        const auto t_begin = now();
        std::vector<uint64_t> part_max(T * 4);
        std::vector<uint8_t> part_ok(T * 4, 1);
        int used = 0;
        bool failed = false;
        for (int c = 0; c < kChunks && !failed && !stop.load(); ++c) {
            const uint64_t qa = c0[c], qb = c0[c + 1], Qc = qb - qa;
            if (Qc) {
                const uint8_t *src = q_ranks + q_offsets[qa];
                const uint64_t n_sym = n_sym_c[c];
                const bool is_raw = raw[c];
                // raw chunks on their own H2D stream: a 175 MB copy does not hold up the packed chunk behind it, whose
                // ring slot the packers want back (queueing every raw chunk up front was tried: the raw stream then
                // starves the packed one and the ring stalls -- 64 ms against 54)
                cudaStream_t cs = is_raw ? ix->copy_in2 : ix->copy_in;
                int slot = 0;
                auto t0 = now();
                if (is_raw) {
                    // the ranks first: the copy engine moves them while the host threads compute this chunk's lengths
                    if (n_sym) cudaMemcpyAsync(d_in[c], src, n_sym, cudaMemcpyHostToDevice, cs);
                    h2d += n_sym;
                } else {
                    slot = used++ % kRing;
                    if (used > kRing) cudaEventSynchronize(ev_slot[slot]);  // the slot's previous H2D has left the staging buffer
                    t_slot += since(t0);
                    t0 = now();
                    std::fill(part_ok.begin(), part_ok.end(), 1);
                }
                uint64_t *dst = h_words[slot];
                pool.run(T * 4, [&, qa, qb, src, n_sym, dst, is_raw](unsigned t) {
                    part_max[t] = kb::query_lengths_host(q_offsets, qa, qb, h_lens + qa, t, T * 4);
                    if (!is_raw) part_ok[t] = kb::pack_stream_host(src, n_sym, bits, sigma, dst, t, T * 4) ? 1 : 0;
                });
                t_pool += since(t0);
                t0 = now();
                uint64_t mx = 0;
                for (uint64_t v : part_max) mx = std::max(mx, v);
                max_len[c] = mx;
                stride[c] = (uint32_t)std::max<uint64_t>(1, (mx + spw - 1) / spw);
                lens16[c] = mx < 65536;
                if (!is_raw && (!lens16[c] || stride[c] > max_stride)) unsupported = failed = true;
                if (!is_raw)
                    for (uint8_t ok : part_ok)
                        if (!ok) bad_rank = failed = true;
                if (!failed) {
                    if (!is_raw) {
                        dst[n_stream_words[c]] = 0;  // the padding word align_stream_kernel may read
                        cudaMemcpyAsync(d_in[c], dst, (n_stream_words[c] + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, cs);
                        h2d += (n_stream_words[c] + 1) * sizeof(uint64_t);
                    }
                    if (lens16[c]) {
                        cudaMemcpyAsync(d_lens[c], h_lens + qa, Qc * sizeof(uint16_t), cudaMemcpyHostToDevice, cs);
                        h2d += Qc * sizeof(uint16_t);
                    } else {
                        cudaMemcpyAsync(d_off[c], q_offsets + qa, (Qc + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, cs);
                        h2d += (Qc + 1) * sizeof(uint64_t);
                    }
                    cudaEventRecord(ev_in[c], cs);
                    if (!is_raw) cudaEventRecord(ev_slot[slot], cs);
                }
                t_enqueue += since(t0);
            }
            {
                std::lock_guard<std::mutex> lock(mu);
                if (failed) producer_failed = true;
                else produced = c + 1;
            }
            cv.notify_all();
        }
        t_producer = since(t_begin);
    };
    try {
        producer = std::thread(produce);
    } catch (const std::system_error &) {  // no thread to be had: the caller takes the single-copy path
        return cleanup(KMER_B200_ERR_UNSUPPORTED);
    }

    uint64_t base = 0;
    bool ok_so_far = true;
    for (int c = 0; c < kChunks; ++c) {
        {
            const auto t0 = now();
            std::unique_lock<std::mutex> lock(mu);
            cv.wait(lock, [&] { return produced > c || producer_failed; });
            t_wait_chunk += since(t0);
            if (produced <= c) {
                ok_so_far = false;
                break;
            }
        }
        const uint64_t qa = c0[c], qb = c0[c + 1], Qc = qb - qa;
        if (Qc == 0) continue;
        const auto t0 = now();
        cudaStreamWaitEvent(st, ev_in[c], 0);
        if (lens16[c]) {
            // lengths -> chunk-relative offsets: widen, exclusive scan (the total lands in entry Qc)
            widen_lens_kernel<<<(unsigned)((Qc + 255) / 256), 256, 0, st>>>(d_lens[c], Qc, d_off[c]);
            kb::launch_offsets_scan(d_off[c], Qc, d_scan, st);
        } else {
            add_base_kernel<<<(unsigned)((Qc + 1 + 255) / 256), 256, 0, st>>>(d_off[c], Qc + 1, 0 - q_offsets[qa]);
        }
        int s;
        if (raw[c]) {
            s = search_device_impl(ix, (const uint8_t *)d_in[c], d_off[c], Qc, max_len[c], mode, nullptr, 0, kFlavorFull, &chunk_res[c]);
        } else {
            const uint64_t n_out = Qc * stride[c];
            s = dev_alloc(ix, &d_words[c], n_out, false);
            if (s == 0) {
                align_stream_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, st>>>((const uint64_t *)d_in[c], d_off[c], d_lens[c], Qc,
                                                                                    stride[c], bits, d_words[c]);
                PackedQueries pk{d_words[c], d_lens[c], stride[c]};
                s = search_device_impl(ix, nullptr, nullptr, Qc, max_len[c], mode, nullptr, 0, kFlavorFull, &chunk_res[c], &pk);
            }
        }
        if (s != 0) return cleanup(s);
        kmer_b200_result *cr = chunk_res[c];
        if (base) add_base_kernel<<<(unsigned)((Qc + 1 + 255) / 256), 256, 0, st>>>(cr->offsets, Qc + 1, base);
        cudaEventRecord(ev_done[c], st);
        cudaStreamWaitEvent(ix->copy_out, ev_done[c], 0);
        cudaMemcpyAsync(res->offsets + qa, cr->offsets, Qc * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->copy_out);
        cudaMemcpyAsync(res->status + qa, cr->status, Qc, cudaMemcpyDeviceToHost, ix->copy_out);
        base += cr->n_positions;
        t_search += since(t0);
    }
    producer.join();
    if (bad_rank) return cleanup(fail(KMER_B200_ERR_INVALID_RANK, "a query contains a rank >= sigma"));
    if (unsupported || !ok_so_far) return cleanup(KMER_B200_ERR_UNSUPPORTED);  // the caller reruns the batch with every chunk raw
    if (!host_result_positions(res, base)) return cleanup(fail(KMER_B200_ERR_OUT_OF_MEMORY, "host allocation for the positions failed"));
    uint64_t at = 0;
    for (int c = 0; c < kChunks; ++c) {
        if (!chunk_res[c] || !chunk_res[c]->n_positions) continue;
        cudaMemcpyAsync(res->positions + at, chunk_res[c]->positions, chunk_res[c]->n_positions * sizeof(uint32_t),
                        cudaMemcpyDeviceToHost, ix->copy_out);
        at += chunk_res[c]->n_positions;
    }
    cudaError_t e = cudaStreamSynchronize(ix->copy_out);
    res->offsets[Q] = base;
    if (e != cudaSuccess) return cleanup(fail(KMER_B200_ERR_CUDA, std::string("search (D2H): ") + cudaGetErrorString(e)));
    ix->last_h2d = h2d;
    ix->last_d2h = Q * 9 + base * sizeof(uint32_t);
    *out = res;
    const double t_loop = since(t_call);
    const int code = cleanup(0);
    if (trace)
        std::fprintf(stderr, "[kmer_b200 host trace] raw %u %%: producer %.2f (slot wait %.2f | lengths + pack %.2f | enqueue %.2f) | caller: "
                     "wait for chunk %.2f | search %.2f | to last D2H %.2f | with cleanup %.2f ms\n", raw_pct, t_producer, t_slot, t_pool,
                     t_enqueue, t_wait_chunk, t_search, t_loop, since(t_call));
    return code;
}

// The device result dres copied into a new host result: a pinned buffer for each array dres holds (the positions as
// host_result_positions places them), copied on the index's stream with one synchronisation. *d2h = the bytes copied.
static int result_to_host(kmer_b200_index *ix, const kmer_b200_result *dres, kmer_b200_result **out, uint64_t *d2h) {
    kmer_b200_result *res = host_result_new(ix, dres->n_queries);
    bool ok = res && host_result_positions(res, dres->n_positions);
    if (ok) res->n_kmers = dres->n_kmers;
    uint64_t bytes = 0;
    for_each_result_array(*dres, [&](auto array, auto cap, uint64_t n) {
        using T = std::remove_reference_t<decltype(*(dres->*array))>;
        if (!ok || !cap || !(dres->*array)) return;
        if (!(res->*array)) ok = (res->*array = (T *)pinned_get(n * sizeof(T), &(res->*cap))) != nullptr;
        if (ok && n) cudaMemcpyAsync(res->*array, dres->*array, n * sizeof(T), cudaMemcpyDeviceToHost, ix->stream), bytes += n * sizeof(T);
    });
    // also when an allocation failed: the copies already queued finish before their buffers go back to the cache
    const cudaError_t e = cudaStreamSynchronize(ix->stream);
    if (!ok || e != cudaSuccess) {
        cudaGetLastError();
        kmer_b200_result_free(res);
        return ok ? fail(KMER_B200_ERR_CUDA, std::string("result (D2H): ") + cudaGetErrorString(e))
                  : fail(KMER_B200_ERR_OUT_OF_MEMORY, "pinned host allocation failed");
    }
    *d2h = bytes;
    *out = res;
    return KMER_B200_OK;
}

// One copy each way: the batch is staged on the device whole, the request runs there, and the result comes back into
// pinned host buffers. Small exact batches, collections, approximate search and seeding take this path.
static int host_batch(kmer_b200_index *ix, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q, const uint8_t *lut256,
                      BatchRequest req, kmer_b200_result **out) {
    KB_TRY(request_check(ix, q_offsets, &req, out));
    const uint64_t n_sym = q_offsets[Q] - q_offsets[0];
    if (n_sym && !q_ranks) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "q_ranks is null");
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    StagedBatch staged(ix);
    KB_TRY(staged.stage(q_ranks, q_offsets, Q, lut256));
    kmer_b200_result *dres = nullptr;
    KB_TRY(request_run(ix, staged.ranks(q_offsets), staged.d_off, Q, staged.max_len, req, &dres));
    uint64_t d2h = 0;
    const int s = result_to_host(ix, dres, out, &d2h);
    kmer_b200_result_free(dres);
    if (s != 0) return s;
    ix->last_h2d = n_sym + (Q + 1) * sizeof(uint64_t);
    ix->last_d2h = d2h;
    ix->last_host_path = 0, ix->last_raw_pct = 100, ix->last_pack_gbs = 0;
    return KMER_B200_OK;
}

static int search_batch_host(kmer_b200_index *ix, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q,
                             uint32_t mode, const uint8_t *lut256, kmer_b200_result **out) {
    if (!ix || !out || !q_offsets) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    if (!ix->replicas.empty()) return search_batch_multi(ix, q_ranks, q_offsets, Q, mode, lut256, out);
    const uint64_t n_sym = q_offsets[Q] - q_offsets[0];
    if (n_sym && !q_ranks) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "q_ranks is null");
    // batches whose transfer dominates (>= 256 MiB over PCIe) are pipelined in chunks
    if (!lut256 && ix->starts.empty() && Q >= (1u << 18) && n_sym + Q * 17 >= (256ull << 20) && !std::getenv("KMER_B200_NO_PIPELINE")) {
        DeviceGuard guard(ix->device);
        std::lock_guard<std::mutex> lock(ix->mu);
        // The share of raw chunks. Pageable input cannot be DMA-ed directly (the driver would stage it at a fraction of the
        // link rate): every chunk is packed straight out of the caller's memory into a pinned ring. Pinned input of 2- and
        // 4-bit alphabets: the share comes from the host's streaming pack rate, measured once per process on the first
        // large batch (other processes sharing the cores -- one per GPU under torchrun -- lower the rate and so raise the
        // share). Pinned input of 8-bit alphabets: packing saves no link bytes, every chunk travels raw.
        cudaPointerAttributes attr{};
        const bool pageable = cudaPointerGetAttributes(&attr, q_ranks) != cudaSuccess || attr.type == cudaMemoryTypeUnregistered;
        cudaGetLastError();
        uint32_t raw_pct = 0;
        double rate = 0;
        if (!pageable && ix->bits == 8) {
            raw_pct = 100;
        } else if (!pageable) {
            rate = stream_pack_rate(q_ranks + q_offsets[0], n_sym, ix->bits, ix->sigma);
            raw_pct = raw_chunk_percent(rate / std::max(1u, ix->host_sharers), ix->bits, n_sym, Q);
        }
        if (const char *env = std::getenv("KMER_B200_HOST_RAW_PCT")) raw_pct = (uint32_t)std::max(0, std::min(100, std::atoi(env)));
        int s = search_batch_host_chunked(ix, q_ranks, q_offsets, Q, mode, raw_pct, out);
        if (s == KMER_B200_ERR_UNSUPPORTED && raw_pct < 100) {  // a packed chunk refused its queries: every chunk raw
            raw_pct = 100;
            s = search_batch_host_chunked(ix, q_ranks, q_offsets, Q, mode, raw_pct, out);
        }
        if (s != KMER_B200_ERR_UNSUPPORTED) {
            ix->last_host_path = 3, ix->last_raw_pct = raw_pct, ix->last_pack_gbs = rate / 1e9;
            return s;
        }
        // no producer thread to be had: one copy each way
    }
    return host_batch(ix, q_ranks, q_offsets, Q, lut256, BatchRequest::exact(mode, kFlavorFull), out);
}

int kmer_b200_search_batch(kmer_b200_index *ix, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q,
                           uint32_t mode, kmer_b200_result **out) {
    return search_batch_host(ix, q_ranks, q_offsets, Q, mode, nullptr, out);
}

int kmer_b200_search_approx_batch(kmer_b200_index *ix, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q,
                                  uint32_t max_mismatches, kmer_b200_result **out) {
    const kmer_b200_approx_options opt{max_mismatches, KMER_B200_HITS_ALL, 0, 0};
    return host_batch(ix, q_ranks, q_offsets, Q, nullptr, BatchRequest::approx(&opt, kFlavorFull), out);
}

int kmer_b200_search_approx_batch_ex(kmer_b200_index *ix, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q,
                                     const kmer_b200_approx_options *opt, kmer_b200_result **out) {
    return host_batch(ix, q_ranks, q_offsets, Q, nullptr, BatchRequest::approx(opt, kFlavorFull), out);
}

int kmer_b200_seed_batch(kmer_b200_index *ix, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q, uint32_t k,
                         uint32_t max_occ, kmer_b200_result **out) {
    return host_batch(ix, q_ranks, q_offsets, Q, nullptr, BatchRequest::seeds(k, max_occ, kFlavorFull), out);
}

int kmer_b200_record_votes(kmer_b200_index *ix, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q, uint32_t k,
                           uint32_t max_occ, uint32_t min_votes, kmer_b200_result **out) {
    return host_batch(ix, q_ranks, q_offsets, Q, nullptr, BatchRequest::votes(k, max_occ, min_votes), out);
}

int kmer_b200_search_batch_ptrs(kmer_b200_index *ix, const uint8_t *const *q_ptrs, const uint64_t *q_lens, uint64_t Q,
                                uint32_t mode, kmer_b200_result **out) {
    if (!ix || !out || (Q && (!q_ptrs || !q_lens))) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    // gather into one buffer with the host threads (offsets by a two-level prefix sum), then the ordinary host batch
    kb::HostPool &pool = kb::HostPool::instance();
    const unsigned T = std::max(1u, pool.threads());
    std::vector<uint64_t> part_sum(T + 1, 0);
    pool.run(T, [&](unsigned t) {
        uint64_t s = 0;
        for (uint64_t i = Q * t / T; i < Q * (t + 1) / T; ++i) s += q_lens[i];
        part_sum[t + 1] = s;
    });
    for (unsigned t = 0; t < T; ++t) part_sum[t + 1] += part_sum[t];
    const uint64_t total = part_sum[T];
    // both buffers are first touched by the threads that fill them (a zero-initialised vector of 10^8 offsets would be
    // 0.8 GB of page faults on the calling thread)
    uint64_t *offsets = (uint64_t *)std::malloc((Q + 1) * sizeof(uint64_t));
    uint8_t *ranks = (uint8_t *)std::malloc(std::max<uint64_t>(total, 1) + 8);
    if (!ranks || !offsets) {
        std::free(offsets);
        std::free(ranks);
        return fail(KMER_B200_ERR_OUT_OF_MEMORY, "host allocation failed");
    }
    bool null_query = false;
    pool.run(T, [&](unsigned t) {
        uint64_t o = part_sum[t];
        const uint64_t i_end = Q * (t + 1) / T;
        for (uint64_t i = Q * t / T; i < i_end; ++i) {
            // the queries are heap blocks of their own: a cache miss each unless asked for ahead of time
            if (i + 16 < i_end && q_ptrs[i + 16]) {
                __builtin_prefetch(q_ptrs[i + 16]);
                __builtin_prefetch(q_ptrs[i + 16] + 63);
            }
            offsets[i] = o;
            if (q_lens[i]) {
                if (!q_ptrs[i]) {
                    null_query = true;
                    continue;
                }
                std::memcpy(ranks + o, q_ptrs[i], q_lens[i]);
            }
            o += q_lens[i];
        }
    });
    offsets[Q] = total;
    int s = null_query ? fail(KMER_B200_ERR_INVALID_ARGUMENT, "a query pointer is null")
                       : search_batch_host(ix, ranks, offsets, Q, mode, nullptr, out);
    std::free(ranks);
    std::free(offsets);
    return s;
}

int kmer_b200_search_batch_text(kmer_b200_index *ix, const char *q_chars, const uint64_t *q_offsets, uint64_t Q,
                                const uint8_t *lut256, uint32_t mode, kmer_b200_result **out) {
    if (!lut256) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "lut256 is null");
    return search_batch_host(ix, reinterpret_cast<const uint8_t *>(q_chars), q_offsets, Q, mode, lut256, out);
}

int kmer_b200_create_from_text(const char *text, uint64_t n, const uint8_t *lut256, uint32_t sigma, const uint32_t *ks,
                               uint32_t n_ks, const kmer_b200_config *cfg, kmer_b200_index **out) {
    if (!lut256) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "lut256 is null");
    if (cfg && cfg->n_devices > 1) return create_multi(reinterpret_cast<const uint8_t *>(text), n, sigma, ks, n_ks, cfg, out, lut256);
    return create_impl(reinterpret_cast<const uint8_t *>(text), false, n, sigma, ks, n_ks, cfg, out, lut256);
}

uint64_t kmer_b200_result_n_queries(const kmer_b200_result *r) { return r ? r->n_queries : 0; }
uint64_t kmer_b200_result_n_positions(const kmer_b200_result *r) { return r ? r->n_positions : 0; }
int kmer_b200_result_on_device(const kmer_b200_result *r) { return r && r->on_device; }
const uint32_t *kmer_b200_result_hit_queries(const kmer_b200_result *r) { return (r && r->on_device) ? r->hit_queries : nullptr; }
const uint64_t *kmer_b200_result_offsets(const kmer_b200_result *r) { return r ? r->offsets : nullptr; }
const uint32_t *kmer_b200_result_positions(const kmer_b200_result *r) { return r ? r->positions : nullptr; }
const uint8_t *kmer_b200_result_status(const kmer_b200_result *r) { return r ? r->status : nullptr; }
const uint8_t *kmer_b200_result_distances(const kmer_b200_result *r) { return r ? r->distances : nullptr; }
const uint8_t *kmer_b200_result_best_distances(const kmer_b200_result *r) { return r ? r->best_distance : nullptr; }
const uint32_t *kmer_b200_result_seed_offsets(const kmer_b200_result *r) { return r ? r->seed_offsets : nullptr; }
const uint32_t *kmer_b200_result_kmer_counts(const kmer_b200_result *r) { return r ? r->kmer_counts : nullptr; }
uint64_t kmer_b200_result_n_kmers(const kmer_b200_result *r) { return r ? r->n_kmers : 0; }
const uint32_t *kmer_b200_result_votes(const kmer_b200_result *r) { return r ? r->votes : nullptr; }
const uint32_t *kmer_b200_result_kmer_hits(const kmer_b200_result *r) { return r ? r->kmer_hits : nullptr; }

void kmer_b200_result_free(kmer_b200_result *r) {
    if (!r) return;
    kmer_b200_index *ix = r->index;
    if (r->on_device) {
        DeviceGuard guard(ix->device);
        for_each_result_array(*r, [&](auto array, auto, uint64_t) { dev_free(ix, r->*array); });
    } else {
        if (r->positions_pageable) {
            std::free(r->positions);
            r->positions = nullptr;
        }
        for_each_result_array(*r, [&](auto array, auto cap, uint64_t) {
            if (cap) pinned_put(r->*array, r->*cap);
        });
    }
    delete r;
}

uint32_t kmer_b200_n_elements(const kmer_b200_index *ix) { return ix ? (uint32_t)primary(ix)->ks.size() : 0; }

int kmer_b200_element_info_get(const kmer_b200_index *ix, uint32_t e, kmer_b200_element_info *out) {
    ix = primary(ix);
    if (!ix || !out || e >= ix->elems.size()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad element");
    const HostElement &he = ix->elems[e];
    out->k = he.dev.k;
    out->key_bits = he.key_bits;
    out->directory_shift = he.dev.shift;
    out->sort_passes = he.sort_passes;
    out->n_kmers = he.dev.n_kmers;
    out->directory_entries = he.dev.dir_entries;
    out->device_bytes = he.bytes;
    if (he.view) {  // a prefix view of the largest k's arrays: it owns nothing
        out->directory_shift = 0;
        out->n_kmers = ix->n - he.dev.k + 1;
        out->directory_entries = 0;
    }
    return KMER_B200_OK;
}

static int reject_view(const kmer_b200_index *ix, uint32_t e) {
    if (e < ix->elems.size() && ix->elems[e].view)
        return fail(KMER_B200_ERR_UNSUPPORTED, "element is a view of the largest k's arrays (shared-positions index)");
    if (e < ix->elems.size() && ix->elems[e].in_parts)
        return fail(KMER_B200_ERR_UNSUPPORTED, "the element's positions live in per-GPU parts (peer-positions index)");
    return 0;
}

int kmer_b200_element_positions(kmer_b200_index *ix, uint32_t e, uint32_t *out, uint64_t cap) {
    ix = primary(ix);
    if (!ix || !out || e >= ix->elems.size()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad element");
    KB_TRY(reject_view(ix, e));
    DeviceGuard guard(ix->device);
    const uint64_t n = std::min<uint64_t>(cap, ix->elems[e].dev.n_kmers);
    KB_CUDA(cudaMemcpyAsync(out, ix->elems[e].d_pos, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ix->stream));
    KB_CUDA(cudaStreamSynchronize(ix->stream));
    return KMER_B200_OK;
}

int kmer_b200_element_hashes(kmer_b200_index *ix, uint32_t e, uint64_t *out, uint64_t cap) {
    ix = primary(ix);
    if (!ix || !out || e >= ix->elems.size()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad element");
    KB_TRY(reject_view(ix, e));
    DeviceGuard guard(ix->device);
    const HostElement &he = ix->elems[e];
    const uint64_t n = std::min<uint64_t>(cap, he.dev.n_kmers);
    if (!he.d_keys) {  // dense directory: the sorted hashes are not kept; recompute them from the text at pos[i]
        uint64_t *d_tmp = nullptr;
        KB_TRY(dev_alloc(ix, &d_tmp, n, false));
        if (n)
            hashes_from_text_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ix->stream>>>(
                kb::PackedText{ix->d_text, ix->n, ix->bits, ix->sigma}, he.dev.k, he.d_pos, n, d_tmp);
        cudaError_t e = cudaMemcpyAsync(out, d_tmp, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ix->stream);
        dev_free(ix, d_tmp);
        if (e != cudaSuccess) return fail(KMER_B200_ERR_CUDA, cudaGetErrorString(e));
        return KMER_B200_OK;
    }
    if (he.key_bytes == 8) {
        KB_CUDA(cudaMemcpyAsync(out, he.d_keys, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->stream));
        KB_CUDA(cudaStreamSynchronize(ix->stream));
    } else {  // widen 32-bit hashes on the host
        std::vector<uint32_t> tmp(n);
        KB_CUDA(cudaMemcpyAsync(tmp.data(), he.d_keys, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ix->stream));
        KB_CUDA(cudaStreamSynchronize(ix->stream));
        for (uint64_t i = 0; i < n; ++i) out[i] = tmp[i] + he.dev.key_lo;
    }
    return KMER_B200_OK;
}

int kmer_b200_element_part(const kmer_b200_index *ix, uint32_t e, kmer_b200_part *out) {
    ix = primary(ix);
    if (!ix || !out || e >= ix->ks.size()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad element");
    KB_TRY(reject_view(ix, e));
    const HostElement &he = ix->elems[e];
    if (he.dev.shift != 0) return fail(KMER_B200_ERR_UNSUPPORTED, "parts are exported from dense directories only");
    out->key_lo = he.dev.key_lo;
    out->key_hi = he.dev.key_hi == UINT64_MAX ? he.dev.key_space : he.dev.key_hi;
    out->n_kmers = he.dev.n_kmers;
    out->directory_entries = he.dev.dir_entries;
    out->d_positions = he.d_pos;
    out->d_directory = he.d_dir;
    return KMER_B200_OK;
}

int kmer_b200_export_directory(kmer_b200_index *ix, uint32_t e, uint64_t base, uint64_t n, uint32_t *d_dst) {
    ix = primary(ix);
    if (!ix || !d_dst || e >= ix->ks.size() || n > ix->elems[e].dev.dir_entries)
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    KB_TRY(reject_view(ix, e));
    DeviceGuard guard(ix->device);
    if (n) add_base32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ix->stream>>>(ix->elems[e].d_dir, n, (uint32_t)base, d_dst);
    KB_CUDA(cudaGetLastError());
    return KMER_B200_OK;
}

int kmer_b200_export_bucket_sizes(kmer_b200_index *ix, uint32_t e, uint8_t *d_sizes, uint64_t *n_large_out) {
    ix = primary(ix);
    if (!ix || !d_sizes || !n_large_out || e >= ix->ks.size()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    KB_TRY(reject_view(ix, e));
    const HostElement &he = ix->elems[e];
    if (he.dev.shift != 0) return fail(KMER_B200_ERR_UNSUPPORTED, "bucket sizes are exported from dense directories only");
    DeviceGuard guard(ix->device);
    unsigned long long *d_large = nullptr;
    KB_TRY(dev_alloc(ix, &d_large, 1, false));
    cudaMemsetAsync(d_large, 0, sizeof(unsigned long long), ix->stream);
    kb::launch_bucket_sizes(he.d_dir, he.dev.dir_entries - 1, d_sizes, d_large, ix->stream);
    unsigned long long large = 0;
    KB_CUDA(cudaMemcpyAsync(&large, d_large, sizeof(large), cudaMemcpyDeviceToHost, ix->stream));
    KB_CUDA(cudaStreamSynchronize(ix->stream));
    dev_free(ix, d_large);
    *n_large_out = large;
    return KMER_B200_OK;
}

int kmer_b200_directory_from_sizes(kmer_b200_index *ix, const uint8_t *d_sizes, uint64_t n_keys, uint32_t *d_directory) {
    ix = primary(ix);
    if (!ix || !d_sizes || !d_directory) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    DeviceGuard guard(ix->device);
    const uint64_t tiles = kb::sizes_tiles(n_keys + 1);  // one entry more than hashes: the sizes array is read as n_keys + 1 with a zero tail
    uint64_t *d_tile = nullptr, *d_sums = nullptr;
    KB_TRY(dev_alloc(ix, &d_tile, tiles + 1, false));
    KB_TRY(dev_alloc(ix, &d_sums, kb::offsets_scan_blocks(tiles) + 1, false));
    kb::launch_sizes_tile_sums(d_sizes, n_keys, d_tile, ix->stream);
    if (kb::sizes_tiles(n_keys) < tiles) cudaMemsetAsync(d_tile + kb::sizes_tiles(n_keys), 0, sizeof(uint64_t), ix->stream);
    kb::launch_offsets_scan(d_tile, tiles, d_sums, ix->stream);
    kb::launch_sizes_to_dir(d_sizes, n_keys, d_tile, d_directory, ix->stream);
    // the sentinel entry d_directory[n_keys] = total
    KB_CUDA(cudaMemcpyAsync(d_directory + n_keys, d_tile + tiles, sizeof(uint32_t), cudaMemcpyDeviceToDevice, ix->stream));
    dev_free(ix, d_tile);
    dev_free(ix, d_sums);
    KB_CUDA(cudaGetLastError());
    return KMER_B200_OK;
}

static int adopt_element_impl(kmer_b200_index *ix, uint32_t e, const uint32_t *d_positions, uint64_t n_kmers,
                              const uint32_t *d_directory, uint64_t directory_entries, int ownership) {
    if (!ix || !d_positions || !d_directory || e >= ix->ks.size()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    if (ix->cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS) return fail(KMER_B200_ERR_UNSUPPORTED, "adopt: not on a shared-positions index");
    HostElement &he = ix->elems[e];
    if (n_kmers != ix->n - he.dev.k + 1 || directory_entries != he.dev.key_space + 1)
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "adopt: array sizes do not describe the whole index (n - k + 1 positions, sigma^k + 1 directory entries)");
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    if (he.adopted != 1) {
        dev_free(ix, he.d_dir);
        dev_free(ix, he.d_pos);
        ix->device_bytes -= he.bytes;
    }
    dev_free(ix, (uint8_t *)he.d_keys);
    he.d_keys = nullptr;
    he.adopted = ownership;
    he.d_pos = const_cast<uint32_t *>(d_positions);
    he.d_dir = const_cast<uint32_t *>(d_directory);
    he.dev.shift = 0;
    he.dev.n_kmers = n_kmers;
    he.dev.dir_entries = directory_entries;
    he.dev.dir = he.d_dir;
    he.dev.keys = nullptr;
    he.dev.pos = he.d_pos;
    he.dev.key_lo = 0;
    he.dev.key_hi = UINT64_MAX;
    he.bytes = n_kmers * 4 + directory_entries * 4;
    if (ownership == 2) ix->device_bytes += he.bytes;
    ix->host_index.elem[e] = he.dev;
    bool all = true;
    for (size_t i = 0; i < ix->ks.size(); ++i) all = all && ix->elems[i].adopted != 0;
    if (all) {
        // the index is whole again: elements built from now on (auxiliary k' = m elements) cover the whole key space;
        // those built for the part are dropped
        ix->cfg.key_parts = 0;
        ix->cfg.key_part = 0;
        for (size_t i = ix->ks.size(); i < ix->elems.size(); ++i) {
            dev_free(ix, ix->elems[i].d_dir);
            dev_free(ix, ix->elems[i].d_pos);
            dev_free(ix, (uint8_t *)ix->elems[i].d_keys);
        }
        ix->elems.resize(ix->ks.size());
        std::memset(ix->host_index.aux_for_len, 0xFF, sizeof(ix->host_index.aux_for_len));
    }
    KB_CUDA(cudaMemcpyAsync(ix->d_index, &ix->host_index, sizeof(kb::DeviceIndex), cudaMemcpyHostToDevice, ix->stream));
    KB_CUDA(cudaStreamSynchronize(ix->stream));
    return KMER_B200_OK;
}

int kmer_b200_adopt_element(kmer_b200_index *ix, uint32_t e, const uint32_t *d_positions, uint64_t n_kmers,
                            const uint32_t *d_directory, uint64_t directory_entries) {
    if (ix && !ix->replicas.empty()) return fail(KMER_B200_ERR_UNSUPPORTED, "not available on a multi-device handle");
    return adopt_element_impl(ix, e, d_positions, n_kmers, d_directory, directory_entries, 1);
}

// library_owned: the multi-device handle's own assembly -- the directory was allocated by the library and this index's own
// part (he.d_pos, one of the parts) stays its property; otherwise everything passed belongs to the caller.
static int adopt_parts_impl(kmer_b200_index *ix, uint32_t e, const uint32_t *const *d_position_parts, const uint64_t *part_first,
                            uint32_t n_parts, const uint32_t *d_directory, uint64_t directory_entries, bool library_owned) {
    if (!ix || !d_position_parts || !part_first || !d_directory || e >= ix->ks.size())
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    if (ix->cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS) return fail(KMER_B200_ERR_UNSUPPORTED, "adopt: not on a shared-positions index");
    if (n_parts == 0 || n_parts > (uint32_t)kb::kMaxPosParts) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "adopt: 1 to 8 parts");
    HostElement &he = ix->elems[e];
    const uint64_t n_kmers = ix->n - he.dev.k + 1;
    if (part_first[0] != 0 || part_first[n_parts] != n_kmers || directory_entries != he.dev.key_space + 1 || n_kmers > 0xFFFFFFFFull)
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "adopt: the parts do not describe the whole index (n - k + 1 positions, sigma^k + 1 directory entries)");
    for (uint32_t r = 0; r < n_parts; ++r)
        if (part_first[r + 1] < part_first[r] || (part_first[r + 1] > part_first[r] && !d_position_parts[r]))
            return fail(KMER_B200_ERR_INVALID_ARGUMENT, "adopt: part boundaries must ascend and non-empty parts need a pointer");
    DeviceGuard guard(ix->device);
    // parts in other GPUs' memory (mapped into this process by the caller, e.g. CUDA IPC): this device must be allowed
    // to read them from a kernel
    for (uint32_t r = 0; r < n_parts; ++r) {
        if (part_first[r + 1] == part_first[r]) continue;
        cudaPointerAttributes attr{};
        if (cudaPointerGetAttributes(&attr, d_position_parts[r]) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
            cudaGetLastError();
            return fail(KMER_B200_ERR_INVALID_ARGUMENT, "adopt: a part is not device memory");
        }
        if (attr.device == ix->device) continue;
        // (memory opened with kmer_b200_peer_buffer_open is readable already; this covers parts on other devices of
        // THIS process)
        int can = 0;
        cudaDeviceCanAccessPeer(&can, ix->device, attr.device);
        if (!can) return fail(KMER_B200_ERR_UNSUPPORTED, "adopt: this device cannot read the device that holds a part");
        const cudaError_t pe = cudaDeviceEnablePeerAccess(attr.device, 0);
        if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) {
            cudaGetLastError();
            return fail(KMER_B200_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(pe));
        }
        cudaGetLastError();
    }
    std::lock_guard<std::mutex> lock(ix->mu);
    if (he.adopted != 1) {
        dev_free(ix, he.d_dir);
        if (!library_owned) dev_free(ix, he.d_pos);
        ix->device_bytes -= he.bytes;
    }
    dev_free(ix, (uint8_t *)he.d_keys);
    he.d_keys = nullptr;
    he.adopted = library_owned ? 2 : 1;
    he.in_parts = true;
    if (!library_owned) he.d_pos = nullptr;  // (library_owned: still this index's part, freed with the index)
    he.d_dir = const_cast<uint32_t *>(d_directory);
    he.dev.shift = 0;
    he.dev.n_kmers = n_kmers;
    he.dev.dir_entries = directory_entries;
    he.dev.dir = he.d_dir;
    he.dev.keys = nullptr;
    he.dev.pos = nullptr;
    he.dev.key_lo = 0;
    he.dev.key_hi = UINT64_MAX;
    he.dev.n_pos_parts = n_parts;
    for (uint32_t r = 0; r <= n_parts; ++r) he.dev.part_first[r] = (uint32_t)part_first[r];
    for (uint32_t r = 0; r < n_parts; ++r) he.dev.pos_part[r] = d_position_parts[r];
    he.bytes = directory_entries * 4;
    if (library_owned) {
        for (uint32_t r = 0; r < n_parts; ++r)
            if (d_position_parts[r] == he.d_pos) he.bytes += (part_first[r + 1] - part_first[r]) * 4;
        ix->device_bytes += he.bytes;
    }
    ix->host_index.elem[e] = he.dev;
    bool all = true;
    for (size_t i = 0; i < ix->ks.size(); ++i) all = all && ix->elems[i].adopted != 0;
    if (all) {
        ix->cfg.key_parts = 0;
        ix->cfg.key_part = 0;
        for (size_t i = ix->ks.size(); i < ix->elems.size(); ++i) {
            dev_free(ix, ix->elems[i].d_dir);
            dev_free(ix, ix->elems[i].d_pos);
            dev_free(ix, (uint8_t *)ix->elems[i].d_keys);
        }
        ix->elems.resize(ix->ks.size());
        std::memset(ix->host_index.aux_for_len, 0xFF, sizeof(ix->host_index.aux_for_len));
    }
    KB_CUDA(cudaMemcpyAsync(ix->d_index, &ix->host_index, sizeof(kb::DeviceIndex), cudaMemcpyHostToDevice, ix->stream));
    KB_CUDA(cudaStreamSynchronize(ix->stream));
    return KMER_B200_OK;
}

int kmer_b200_adopt_element_parts(kmer_b200_index *ix, uint32_t e, const uint32_t *const *d_position_parts,
                                  const uint64_t *part_first, uint32_t n_parts, const uint32_t *d_directory,
                                  uint64_t directory_entries) {
    if (ix && !ix->replicas.empty()) return fail(KMER_B200_ERR_UNSUPPORTED, "not available on a multi-device handle");
    return adopt_parts_impl(ix, e, d_position_parts, part_first, n_parts, d_directory, directory_entries, false);
}

// ---- device buffers shared between processes (one process per GPU): what the peer-positions index reads over NVLink --
int kmer_b200_peer_buffer_create(int device, uint64_t bytes, void **d_ptr, uint8_t *handle64) {
    if (!d_ptr || !handle64) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    DeviceGuard guard(device);
    void *p = nullptr;
    // A plain allocation (pool memory cannot be exported) whose size is a multiple of 2 MiB: measured on B200
    // (profiles/tools/ipc_probe.py), an imported allocation of any other size is mapped with small pages and random reads
    // from it run at 0.1 G/s instead of 6.8 G/s.
    bytes = (std::max<uint64_t>(bytes, 1) + (2u << 20) - 1) / (2u << 20) * (2u << 20);
    KB_CUDA(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    const cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaFree(p);
        return fail(KMER_B200_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
    }
    std::memcpy(handle64, &h, 64);
    *d_ptr = p;
    return KMER_B200_OK;
}

int kmer_b200_peer_buffer_open(int device, const uint8_t *handle64, void **d_ptr) {
    if (!d_ptr || !handle64) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    DeviceGuard guard(device);  // mapped into the context of the device whose kernels will read it
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle64, 64);
    void *p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(KMER_B200_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
    }
    *d_ptr = p;
    return KMER_B200_OK;
}

int kmer_b200_peer_buffer_release(int device, void *d_ptr, int opened) {
    if (!d_ptr) return KMER_B200_OK;
    DeviceGuard guard(device);
    cudaDeviceSynchronize();
    const cudaError_t e = opened ? cudaIpcCloseMemHandle(d_ptr) : cudaFree(d_ptr);
    cudaGetLastError();
    return e == cudaSuccess ? KMER_B200_OK : fail(KMER_B200_ERR_CUDA, cudaGetErrorString(e));
}

// ---- FASTA / FASTQ parsing (fastx_kernels.cu) ---------------------------------------------------------------------
struct kmer_b200_records {
    int device = 0;
    uint8_t *d_ranks = nullptr;
    uint64_t n_symbols = 0;
    std::vector<uint64_t> starts;          // [count + 1]
    std::vector<uint64_t> header_offsets;  // [count]
};

int kmer_b200_parse_sequences(const char *data, uint64_t n_bytes, const uint8_t *lut256, uint32_t sigma, uint32_t format,
                              const kmer_b200_config *cfg, kmer_b200_records **out) {
    if (!data || !lut256 || !out || format > 2 || sigma < 2 || sigma > 256) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    *out = nullptr;
    if (n_bytes == 0) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "empty input");
    if (format == 0) format = data[0] == '@' ? 2 : 1;
    int device = cfg ? cfg->device : -1;
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) {
        cudaGetLastError();
        return fail(KMER_B200_ERR_CUDA, "no usable CUDA device (libkmer_b200 has no CPU fallback)");
    }
    DeviceGuard guard(device);
    cudaStream_t st = cfg && cfg->stream ? (cudaStream_t)cfg->stream : nullptr;
    const uint64_t tiles = kb::fastx_tiles(n_bytes);
    uint8_t *d_data = nullptr, *d_lut = nullptr, *d_ranks = nullptr;
    uint64_t *d_nl = nullptr, *d_kept = nullptr, *d_recs = nullptr, *d_sums = nullptr, *d_rec_sym = nullptr, *d_rec_hdr = nullptr;
    int64_t *d_last = nullptr;
    uint32_t *d_err = nullptr;
    auto release = [&](int code) {
        kb_free_async(d_data, st);
        kb_free_async(d_lut, st);
        kb_free_async(d_nl, st);
        kb_free_async(d_kept, st);
        kb_free_async(d_recs, st);
        kb_free_async(d_sums, st);
        kb_free_async(d_rec_sym, st);
        kb_free_async(d_rec_hdr, st);
        kb_free_async(d_last, st);
        kb_free_async(d_err, st);
        if (code != 0) kb_free_async(d_ranks, st);
        cudaStreamSynchronize(st);
        cudaGetLastError();
        return code;
    };
#define KB_FX(expr)                                                                                                        \
    do {                                                                                                                   \
        cudaError_t _e = (expr);                                                                                           \
        if (_e != cudaSuccess) {                                                                                           \
            cudaGetLastError();                                                                                            \
            return release(fail(_e == cudaErrorMemoryAllocation ? KMER_B200_ERR_OUT_OF_MEMORY : KMER_B200_ERR_CUDA,        \
                                std::string(#expr) + ": " + cudaGetErrorString(_e)));                                      \
        }                                                                                                                  \
    } while (0)
    KB_FX(kb_malloc_async((void **)&d_data, n_bytes, st));
    KB_FX(kb_malloc_async((void **)&d_lut, 256, st));
    KB_FX(kb_malloc_async((void **)&d_nl, (tiles + 1) * 8, st));
    KB_FX(kb_malloc_async((void **)&d_kept, (tiles + 1) * 8, st));
    KB_FX(kb_malloc_async((void **)&d_recs, (tiles + 1) * 8, st));
    KB_FX(kb_malloc_async((void **)&d_sums, (kb::offsets_scan_blocks(tiles) + 1) * 8, st));
    KB_FX(kb_malloc_async((void **)&d_last, tiles * 8, st));
    KB_FX(kb_malloc_async((void **)&d_err, 4, st));
    KB_FX(cudaMemcpyAsync(d_data, data, n_bytes, cudaMemcpyHostToDevice, st));
    KB_FX(cudaMemcpyAsync(d_lut, lut256, 256, cudaMemcpyHostToDevice, st));
    KB_FX(cudaMemsetAsync(d_err, 0, 4, st));
    kb::launch_fastx_tile_stats(d_data, n_bytes, d_nl, d_last, st);
    kb::launch_offsets_scan(d_nl, tiles, d_sums, st);  // -> line feeds before each tile
    kb::launch_fastx_count(d_data, n_bytes, format, d_nl, d_last, d_kept, d_recs, st);
    kb::launch_offsets_scan(d_kept, tiles, d_sums, st);
    kb::launch_offsets_scan(d_recs, tiles, d_sums, st);
    uint64_t totals[2] = {0, 0};
    KB_FX(cudaMemcpyAsync(&totals[0], d_kept + tiles, 8, cudaMemcpyDeviceToHost, st));
    KB_FX(cudaMemcpyAsync(&totals[1], d_recs + tiles, 8, cudaMemcpyDeviceToHost, st));
    KB_FX(cudaStreamSynchronize(st));
    const uint64_t n_sym = totals[0], n_rec = totals[1];
    KB_FX(kb_malloc_async((void **)&d_ranks, std::max<uint64_t>(n_sym, 1), st));
    KB_FX(kb_malloc_async((void **)&d_rec_sym, std::max<uint64_t>(n_rec, 1) * 8, st));
    KB_FX(kb_malloc_async((void **)&d_rec_hdr, std::max<uint64_t>(n_rec, 1) * 8, st));
    kb::launch_fastx_write(d_data, n_bytes, format, d_nl, d_last, d_kept, d_recs, d_lut, sigma, d_ranks, d_rec_sym, d_rec_hdr, d_err, st);
    kmer_b200_records *r = new (std::nothrow) kmer_b200_records();
    if (!r) return release(fail(KMER_B200_ERR_OUT_OF_MEMORY, "host allocation failed"));
    std::vector<uint64_t> sym(n_rec), hdr(n_rec);
    uint32_t err = 0;
    cudaError_t e = cudaSuccess;
    if (n_rec) {
        e = cudaMemcpyAsync(sym.data(), d_rec_sym, n_rec * 8, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(hdr.data(), d_rec_hdr, n_rec * 8, cudaMemcpyDeviceToHost, st);
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess || (err & 1u)) {
        delete r;
        return release(e != cudaSuccess ? fail(KMER_B200_ERR_CUDA, std::string("parse_sequences: ") + cudaGetErrorString(e))
                                        : fail(KMER_B200_ERR_INVALID_RANK, "a sequence character is not in the alphabet"));
    }
    r->device = device;
    r->d_ranks = d_ranks;
    r->n_symbols = n_sym;
    if (n_rec == 0 || sym[0] > 0) {  // sequence before the first header line: an unnamed first record
        r->starts.push_back(0);
        r->header_offsets.push_back(UINT64_MAX);
    }
    for (uint64_t i = 0; i < n_rec; ++i) {
        r->starts.push_back(sym[i]);
        r->header_offsets.push_back(hdr[i]);
    }
    r->starts.push_back(n_sym);
    *out = r;
    return release(0);
#undef KB_FX
}

uint64_t kmer_b200_records_count(const kmer_b200_records *r) { return r ? r->header_offsets.size() : 0; }
uint64_t kmer_b200_records_symbols(const kmer_b200_records *r) { return r ? r->n_symbols : 0; }
const uint64_t *kmer_b200_records_starts(const kmer_b200_records *r) { return r ? r->starts.data() : nullptr; }
const uint64_t *kmer_b200_records_header_offsets(const kmer_b200_records *r) { return r ? r->header_offsets.data() : nullptr; }
const uint8_t *kmer_b200_records_ranks_device(const kmer_b200_records *r) { return r ? r->d_ranks : nullptr; }

// positions -> (record, offset) by a binary search in the record table s[0..R]; see kmer_b200_records_locate
static void locate_host(const std::vector<uint64_t> &s, const uint32_t *positions, uint64_t n, uint64_t query_len,
                        uint32_t *record_out, uint32_t *offset_out) {
    for (uint64_t i = 0; i < n; ++i) {
        const uint64_t p = positions[i];
        const size_t rec = (size_t)(std::upper_bound(s.begin(), s.end(), p) - s.begin()) - 1;
        if (rec + 1 >= s.size()) {
            record_out[i] = UINT32_MAX;
            offset_out[i] = 0;
            continue;
        }
        record_out[i] = (query_len && p + query_len > s[rec + 1]) ? UINT32_MAX : (uint32_t)rec;
        offset_out[i] = (uint32_t)(p - s[rec]);
    }
}

int kmer_b200_records_locate(const kmer_b200_records *r, const uint32_t *positions, uint64_t n, uint64_t query_len,
                             uint32_t *record_out, uint32_t *offset_out) {
    if (!r || (n && (!positions || !record_out || !offset_out))) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    locate_host(r->starts, positions, n, query_len, record_out, offset_out);
    return KMER_B200_OK;
}

// ---- collection index ----------------------------------------------------------------------------------------------
int kmer_b200_attach_records(kmer_b200_index *ix, const uint64_t *starts, uint64_t n_records) {
    if (!ix || !starts) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    if (n_records == 0 || n_records >= (1ull << 32)) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "n_records must be in [1, 2^32)");
    KB_TRY(whole_index_check(ix, "a collection index"));
    if (!ix->starts.empty()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "records are attached already");
    KB_TRY(records_check(ix, starts, n_records));
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    return attach_records_impl(ix, starts, n_records);
}

const uint64_t *kmer_b200_index_records(const kmer_b200_index *ix, uint64_t *n_records) {
    const bool has = ix && !ix->starts.empty();
    if (n_records) *n_records = has ? ix->starts.size() - 1 : 0;
    return has ? ix->starts.data() : nullptr;
}

int kmer_b200_locate(kmer_b200_index *ix, const uint32_t *positions, uint64_t n, uint32_t *record_out, uint32_t *offset_out) {
    if (!ix || (n && (!positions || !record_out || !offset_out))) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    if (ix->starts.empty()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "the index has no records: kmer_b200_attach_records");
    locate_host(ix->starts, positions, n, 0, record_out, offset_out);
    return KMER_B200_OK;
}

int kmer_b200_locate_device(kmer_b200_index *ix, const uint32_t *d_positions, uint64_t n, uint32_t *d_record_out,
                            uint32_t *d_offset_out) {
    if (!ix || (n && (!d_positions || !d_record_out || !d_offset_out))) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    if (ix->starts.empty()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "the index has no records: kmer_b200_attach_records");
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    kb::launch_locate(ix->d_starts, ix->starts.size() - 1, d_positions, n, d_record_out, d_offset_out, ix->stream);
    KB_CUDA(cudaGetLastError());
    return KMER_B200_OK;
}

// ---- k-mer spectrum (spectrum.cu). The caller of each helper holds the handle's lock and device.

// bins of the histogram behind kmer_b200_frequent_kmers and kmer_b200_occurrence_cutoff: counts up to 65 534 are read off
// it, larger ones (at most n / 65 535 hashes) are selected and sorted
constexpr uint64_t kSpectrumSelectBins = 1ull << 16;
constexpr uint64_t kSpectrumMaxBins = 1ull << 24;

// the element of k (not an auxiliary one; views included), after the handle checks of whole_index_check
static int spectrum_check(const kmer_b200_index *ix, uint32_t k, uint32_t *elem) {
    KB_TRY(whole_index_check(ix, "the k-mer spectrum", true));
    for (size_t e = 0; e < ix->ks.size(); ++e)
        if (ix->ks[e] == k) {
            *elem = (uint32_t)e;
            return KMER_B200_OK;
        }
    return fail(KMER_B200_ERR_INVALID_ARGUMENT, "k-mer spectrum: k is not one of the index's ks");
}

// windows p < s < p + k charged to record start r (no start in (p, s)); the rule of spectrum_corrections_kernel
static uint64_t junction_windows(const std::vector<uint64_t> &starts, uint64_t r, uint64_t n, uint32_t k) {
    const uint64_t s = starts[r], prev = starts[r - 1];
    if (s == 0 || s <= prev) return 0;
    const uint64_t lo = std::max<uint64_t>(s + 1 >= k ? s + 1 - k : 0, prev), hi = std::min<uint64_t>(s - 1, n - k);
    return hi >= lo ? hi - lo + 1 : 0;
}

// One spectrum of one element: the raw sweep of its directory, then the corrections (record junctions of a collection,
// tail starts of a view). Kept for the selections of kmer_b200_frequent_kmers and kmer_b200_occurrence_cutoff.
struct Spectrum {
    kmer_b200_index *ix = nullptr;
    kb::SpectrumArgs a{};
    std::vector<uint64_t> hist;
    uint64_t total = 0, distinct = 0, max_count = 0, key_space = 0;
    ~Spectrum() {
        if (!ix) return;
        dev_free(ix, a.hist);
        dev_free(ix, a.stats);
        dev_free(ix, a.tab_keys);
        dev_free(ix, a.tab_delta);
    }
};

// the hashes with corrected count >= thr, in hash order: *n_sel of them, the largest count *max_sel. d_hashes == null:
// count pass only; else *d_hashes / *d_counts are allocated here and freed by the caller.
static int spectrum_select(Spectrum &sp, uint64_t thr, uint64_t *n_sel, uint64_t *max_sel, uint64_t **d_hashes = nullptr,
                           uint32_t **d_counts = nullptr) {
    kmer_b200_index *ix = sp.ix;
    cudaStream_t st = ix->stream;
    const uint64_t tiles = kb::spectrum_tiles(sp.a.n_items);
    kb::SpectrumSelect sel{thr, nullptr, nullptr, nullptr};
    uint64_t *block_sums = nullptr;
    auto done = [&](int r) {
        dev_free(ix, sel.tile);
        dev_free(ix, block_sums);
        return r;
    };
    if (dev_alloc(ix, &sel.tile, tiles + 1, false) || dev_alloc(ix, &block_sums, kb::offsets_scan_blocks(tiles) + 1, false))
        return done(KMER_B200_ERR_OUT_OF_MEMORY);
    cudaMemsetAsync(sp.a.stats + 3, 0, sizeof(uint64_t), st);
    kb::launch_spectrum_select(sp.a, sel, false, st);
    kb::launch_offsets_scan(sel.tile, tiles, block_sums, st);
    cudaMemcpyAsync(&ix->h_pinned[6], sel.tile + tiles, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(&ix->h_pinned[7], sp.a.stats + 3, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return done(fail(KMER_B200_ERR_CUDA, std::string("k-mer spectrum: ") + cudaGetErrorString(e)));
    *n_sel = ix->h_pinned[6];
    *max_sel = ix->h_pinned[7];
    if (d_hashes) {
        if (dev_alloc(ix, d_hashes, *n_sel, false) || dev_alloc(ix, d_counts, *n_sel, false)) return done(KMER_B200_ERR_OUT_OF_MEMORY);
        sel.hashes = *d_hashes;
        sel.counts = *d_counts;
        kb::launch_spectrum_select(sp.a, sel, true, st);
    }
    return done(KMER_B200_OK);
}

static int spectrum_compute(kmer_b200_index *ix, uint32_t elem, uint64_t n_bins, Spectrum &sp) {
    using namespace kb;
    cudaStream_t st = ix->stream;
    const Element &E = ix->elems[elem].dev;
    sp.ix = ix;
    sp.a.E = E;
    sp.key_space = 1;
    for (uint32_t i = 0; i < E.k; ++i)
        if (__builtin_mul_overflow(sp.key_space, (uint64_t)ix->sigma, &sp.key_space)) {
            sp.key_space = UINT64_MAX;
            break;
        }
    sp.a.source = E.width != 1 ? kSpectrumSlabs : (E.shift == 0 ? kSpectrumDense : kSpectrumRuns);
    sp.a.n_items = sp.a.source == kSpectrumRuns ? E.n_kmers : sp.key_space;
    sp.a.n_bins = (uint32_t)n_bins;
    KB_TRY(dev_alloc(ix, &sp.a.hist, n_bins, false));
    KB_TRY(dev_alloc(ix, &sp.a.stats, 4, false));
    KB_CUDA(cudaMemsetAsync(sp.a.hist, 0, n_bins * sizeof(uint64_t), st));
    KB_CUDA(cudaMemsetAsync(sp.a.stats, 0, 4 * sizeof(uint64_t), st));
    launch_spectrum_sweep(sp.a, st);
    // corrections: every window across a record start (a collection; charged to the first start above it) and the
    // k_phys - k tail starts of a view (a collection is never a shared-positions index)
    const uint64_t R = ix->starts.empty() ? 0 : ix->starts.size() - 1;
    const uint32_t n_tail = E.k_phys - E.k;
    uint64_t n_corr = n_tail;
    for (uint64_t r = 1; r < R; ++r) n_corr += junction_windows(ix->starts, r, ix->n, E.k);
    if (n_corr) {
        uint64_t cap = 64;
        while (cap < 2 * n_corr) cap <<= 1;
        if (cap > (1ull << 32)) return fail(KMER_B200_ERR_UNSUPPORTED, "k-mer spectrum: more than 2^31 windows cross a record start");
        KB_TRY(dev_alloc(ix, &sp.a.tab_keys, cap, false));
        KB_TRY(dev_alloc(ix, &sp.a.tab_delta, cap, false));
        KB_CUDA(cudaMemsetAsync(sp.a.tab_keys, 0xFF, cap * sizeof(uint64_t), st));
        KB_CUDA(cudaMemsetAsync(sp.a.tab_delta, 0, cap * sizeof(int), st));
        sp.a.tab_mask = (uint32_t)(cap - 1);
        sp.a.tail = n_tail ? 1 : 0;
        launch_spectrum_corrections(sp.a, ix->host_index.text, ix->d_starts, R, n_tail, st);
    }
    sp.hist.assign(n_bins, 0);
    uint64_t stats[4] = {};
    KB_CUDA(cudaMemcpyAsync(sp.hist.data(), sp.a.hist, n_bins * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaMemcpyAsync(stats, sp.a.stats, sizeof(stats), cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));
    KB_CUDA(cudaGetLastError());
    sp.distinct = stats[0];
    sp.total = E.n_kmers + stats[2];  // the raw sweep counts the owner's n - k_phys + 1 windows; stats[2] = signed deltas
    sp.hist[0] = sp.key_space == UINT64_MAX ? UINT64_MAX : sp.key_space - sp.distinct;
    sp.max_count = stats[1];
    if (n_corr) {  // a corrected bucket may have held the maximum: read it off the histogram, or select the overflow bin
        sp.max_count = 0;
        for (uint64_t c = n_bins - 2; c >= 1 && !sp.max_count; --c)
            if (sp.hist[c]) sp.max_count = c;
        if (sp.hist[n_bins - 1]) {
            uint64_t n_sel = 0;
            KB_TRY(spectrum_select(sp, n_bins - 1, &n_sel, &sp.max_count));
        }
    }
    return KMER_B200_OK;
}

// the selection of hashes with count >= thr, sorted by count descending then hash ascending; entries [first, first + n)
// to the host arrays (hashes may be null)
static int spectrum_sorted(Spectrum &sp, uint64_t thr, uint64_t first, uint64_t n, uint64_t *hashes, uint64_t *counts, uint64_t *n_sel) {
    kmer_b200_index *ix = sp.ix;
    cudaStream_t st = ix->stream;
    uint64_t max_sel = 0, *d_h = nullptr, *d_out = nullptr;
    uint32_t *d_c = nullptr, *d_keys = nullptr, *d_order = nullptr;
    auto done = [&](int r) {
        dev_free(ix, d_h);
        dev_free(ix, d_c);
        dev_free(ix, d_keys);
        dev_free(ix, d_order);
        dev_free(ix, d_out);
        return r;
    };
    int r = spectrum_select(sp, thr, n_sel, &max_sel, &d_h, &d_c);
    if (r) return done(r);
    if (*n_sel >= (1ull << 32)) return done(fail(KMER_B200_ERR_UNSUPPORTED, "k-mer spectrum: 2^32 or more k-mers selected"));
    n = std::min(n, *n_sel > first ? *n_sel - first : 0);
    if (n == 0) return done(KMER_B200_OK);
    if (max_sel > thr) {  // hash order already; one stable sort by count
        if (dev_alloc(ix, &d_keys, *n_sel, false) || dev_alloc(ix, &d_order, *n_sel, false)) return done(KMER_B200_ERR_OUT_OF_MEMORY);
        kb::launch_spectrum_sort_keys(d_c, *n_sel, (uint32_t)max_sel, d_keys, d_order, st);
        if ((r = sort_pairs_u32(ix, d_keys, &d_order, *n_sel, bit_length(max_sel - thr)))) return done(r);
    }
    if (dev_alloc(ix, &d_out, 2 * n, false)) return done(KMER_B200_ERR_OUT_OF_MEMORY);
    if (d_order)
        kb::launch_spectrum_gather(d_h, d_c, d_order + first, n, d_out, d_out + n, st);
    else
        kb::launch_spectrum_gather(d_h + first, d_c + first, nullptr, n, d_out, d_out + n, st);
    if (hashes) cudaMemcpyAsync(hashes, d_out, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(counts, d_out + n, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return done(fail(KMER_B200_ERR_CUDA, std::string("k-mer spectrum: ") + cudaGetErrorString(e)));
    return done(KMER_B200_OK);
}

int kmer_b200_spectrum(kmer_b200_index *ix, uint32_t k, uint64_t *hist, uint64_t n_bins, kmer_b200_spectrum_info *info) {
    if (!ix) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    if (n_bins < 2 || n_bins > kSpectrumMaxBins) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "k-mer spectrum: n_bins must be in [2, 2^24]");
    uint32_t elem = 0;
    KB_TRY(spectrum_check(ix, k, &elem));
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    Spectrum sp;
    KB_TRY(spectrum_compute(ix, elem, n_bins, sp));
    if (hist) std::memcpy(hist, sp.hist.data(), n_bins * sizeof(uint64_t));
    if (info) *info = kmer_b200_spectrum_info{sp.total, sp.distinct, sp.max_count, sp.key_space};
    return KMER_B200_OK;
}

int kmer_b200_frequent_kmers(kmer_b200_index *ix, uint32_t k, uint64_t min_count, uint64_t *hashes, uint64_t *counts, uint64_t cap,
                             uint64_t *n_out) {
    if (!ix || !n_out || (cap && (!hashes || !counts))) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    if (min_count == 0) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "frequent k-mers: min_count must be >= 1");
    uint32_t elem = 0;
    KB_TRY(spectrum_check(ix, k, &elem));
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    Spectrum sp;
    const uint64_t last = kSpectrumSelectBins - 1;
    KB_TRY(spectrum_compute(ix, elem, kSpectrumSelectBins, sp));
    // threshold c*: the largest count whose tail #{count >= c*} holds the min(N, cap) entries wanted (the histogram is
    // exact below its last bin); above it N itself comes from the selection
    uint64_t thr = min_count, N = 0;
    if (min_count <= last) {
        for (uint64_t c = min_count; c <= last; ++c) N += sp.hist[c];
        const uint64_t want = std::min(N, cap);
        *n_out = N;
        if (want == 0) return KMER_B200_OK;
        uint64_t cum = 0;
        for (uint64_t c = last; c >= min_count; --c)
            if ((cum += sp.hist[c]) >= want) {
                thr = c;
                break;
            }
    }
    uint64_t n_sel = 0;
    KB_TRY(spectrum_sorted(sp, thr, 0, cap, hashes, counts, &n_sel));
    *n_out = min_count <= last ? N : n_sel;
    return KMER_B200_OK;
}

int kmer_b200_occurrence_cutoff(kmer_b200_index *ix, uint32_t k, double fraction, uint64_t *cutoff) {
    if (!ix || !cutoff) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    if (!(fraction >= 0.0 && fraction < 1.0)) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "occurrence cutoff: fraction must be in [0, 1)");
    uint32_t elem = 0;
    KB_TRY(spectrum_check(ix, k, &elem));
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    Spectrum sp;
    const uint64_t last = kSpectrumSelectBins - 1;
    KB_TRY(spectrum_compute(ix, elem, kSpectrumSelectBins, sp));
    *cutoff = 0;
    if (sp.distinct == 0) return KMER_B200_OK;
    // #{count > c} <= F holds exactly from the (F + 1)-th largest count on: the cutoff is that count
    const uint64_t F = (uint64_t)std::floor(fraction * (double)sp.distinct);
    uint64_t cum = 0;
    for (uint64_t c = last; c >= 1; --c) {
        if ((cum += sp.hist[c]) < F + 1) continue;
        if (c < last) {
            *cutoff = c;
            return KMER_B200_OK;
        }
        uint64_t n_sel = 0;
        return spectrum_sorted(sp, last, F, 1, nullptr, cutoff, &n_sel);
    }
    return fail(KMER_B200_ERR_CUDA, "occurrence cutoff: the histogram does not add up to the distinct k-mers");
}

void kmer_b200_records_free(kmer_b200_records *r) {
    if (!r) return;
    DeviceGuard guard(r->device);
    cudaDeviceSynchronize();
    kb_free_async(r->d_ranks, nullptr);
    cudaStreamSynchronize(nullptr);
    cudaGetLastError();
    delete r;
}

// ---- key-range multi-GPU search: routing (route_kernels.cu) -----------------------------------------------------------
static int routable(const kmer_b200_index *ix) {
    if (!ix) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null index");
    if (!ix->replicas.empty()) return fail(KMER_B200_ERR_UNSUPPORTED, "not available on a multi-device handle");
    KB_NOT_ON_COLLECTION(ix);
    if (ix->ks.size() != 1 || ix->elems[0].key_bytes != 4 || ix->elems[0].dev.shift != 0)
        return fail(KMER_B200_ERR_UNSUPPORTED, "query routing needs a single-k index with 32-bit hashes and a dense directory");
    return 0;
}

int kmer_b200_route_plan_make(const kmer_b200_index *ix, uint64_t n_queries, uint64_t max_query_len, uint32_t n_parts, double slack,
                              kmer_b200_route_plan *out) {
    KB_TRY(routable(ix));
    if (!out || n_parts == 0 || n_parts > (uint32_t)kb::kMaxParts) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    const uint32_t spw = 64 / ix->bits;
    const uint64_t stride = std::max<uint64_t>(1, (std::max<uint64_t>(max_query_len, 1) + spw - 1) / spw);
    if (stride > 16 || max_query_len > 65535) return fail(KMER_B200_ERR_UNSUPPORTED, "queries longer than 16 packed words are not routed");
    if (slack <= 0) slack = 1.25;
    const uint64_t cap = (uint64_t)((double)(n_queries / n_parts + 1) * slack) + 1024;
    if (cap >= 0xFFFFFFFFull) return fail(KMER_B200_ERR_UNSUPPORTED, "batch too large: split it");
    out->n_parts = n_parts;
    out->stride = (uint32_t)stride;
    out->capacity = (uint32_t)std::min<uint64_t>(cap, n_queries + 1024);
    out->reserved = 0;
    out->block_bytes = kb::route_block_bytes(out->capacity, out->stride);
    out->return_block_bytes = kb::route_return_block_bytes(out->capacity);
    return KMER_B200_OK;
}

int kmer_b200_route_queries_device(kmer_b200_index *ix, const uint8_t *d_q, const uint64_t *d_off, uint64_t Q, uint32_t mode,
                                   const kmer_b200_route_plan *plan, uint8_t *d_send_blocks, uint8_t *d_status, uint32_t *sent_counts) {
    KB_TRY(routable(ix));
    if (!plan || !d_send_blocks || !sent_counts || (Q && (!d_off || !d_status))) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    if (mode == UINT32_MAX) mode = ix->cfg.mode;
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    cudaStream_t st = ix->stream;
    uint32_t *d_flags = nullptr;
    KB_TRY(dev_alloc(ix, &d_flags, 1, false));
    cudaMemsetAsync(d_flags, 0, sizeof(uint32_t), st);
    KB_CUDA(cudaMemset2DAsync(d_send_blocks, plan->block_bytes, 0, 64, plan->n_parts, st));  // the block headers
    kb::RouteArgs a{};
    a.q_ranks = d_q;
    a.q_offsets = d_off;
    a.n_queries = Q;
    a.mode = mode;
    a.bits = ix->bits;
    a.sigma = ix->sigma;
    a.k = ix->ks[0];
    {
        kmer_b200_config c = ix->cfg;
        c.key_part = 0;
        c.key_parts = plan->n_parts;
        a.part_width = std::max<uint64_t>(1, key_range_of(c, ix->elems[0].dev.key_space).hi);  // part 0's upper bound = the width
    }
    a.n_parts = plan->n_parts;
    a.stride = plan->stride;
    a.capacity = plan->capacity;
    a.blocks = d_send_blocks;
    a.block_bytes = plan->block_bytes;
    a.status = d_status;
    a.flags = d_flags;
    kb::launch_route_pack(a, st);
    uint32_t flags = 0;
    KB_CUDA(cudaMemcpy2DAsync(sent_counts, sizeof(uint32_t), d_send_blocks, plan->block_bytes, sizeof(uint32_t), plan->n_parts,
                              cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaMemcpyAsync(&flags, d_flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));
    dev_free(ix, d_flags);
    KB_CUDA(cudaGetLastError());
    if (flags & 1u) return fail(KMER_B200_ERR_INVALID_RANK, "a query contains a rank >= sigma");
    if (flags & 2u) return fail(KMER_B200_ERR_UNSUPPORTED, "the batch holds a query shorter than k (or longer than the plan's stride): not routable");
    return KMER_B200_OK;  // counts above plan->capacity: the caller re-plans (all ranks together) and routes again
}

int kmer_b200_search_routed_device(kmer_b200_index *ix, uint8_t *d_recv_blocks, const kmer_b200_route_plan *plan, uint32_t mode,
                                   uint8_t *d_return_blocks, uint64_t *position_splits, kmer_b200_result **out) {
    KB_TRY(routable(ix));
    if (!plan || !d_recv_blocks || !d_return_blocks || !position_splits || !out) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    cudaStream_t st = ix->stream;
    const uint32_t N = plan->n_parts;
    uint32_t counts[kb::kMaxParts] = {};
    KB_CUDA(cudaMemcpy2DAsync(counts, sizeof(uint32_t), d_recv_blocks, plan->block_bytes, sizeof(uint32_t), N, cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaStreamSynchronize(st));
    kb::RoutePrefix pfx{};
    for (uint32_t b = 0; b < N; ++b) {
        if (counts[b] > plan->capacity) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "received block with more records than its capacity");
        pfx.p[b + 1] = pfx.p[b] + counts[b];
    }
    const uint64_t Qr = pfx.p[N];
    uint64_t *d_words = nullptr;
    uint16_t *d_lens = nullptr;
    KB_TRY(dev_alloc(ix, &d_words, Qr * plan->stride, false));
    KB_TRY(dev_alloc(ix, &d_lens, Qr, false));
    kb::launch_compact_blocks(d_recv_blocks, plan->block_bytes, N, plan->capacity, plan->stride, pfx, d_words, d_lens, st);
    PackedQueries pk{d_words, d_lens, plan->stride};
    kmer_b200_result *res = nullptr;
    const uint64_t max_len = (uint64_t)plan->stride * (64 / ix->bits);
    int s = search_device_impl(ix, nullptr, nullptr, Qr, max_len, mode, nullptr, 0, kFlavorFull, &res, &pk);
    dev_free(ix, d_words);
    dev_free(ix, d_lens);
    if (s != 0) return s;
    kb::launch_pack_return(res->offsets, res->status, pfx, N, d_return_blocks, plan->return_block_bytes, plan->capacity, st);
    cudaError_t e = cudaMemcpy2DAsync(position_splits, sizeof(uint64_t), d_return_blocks + 8, plan->return_block_bytes, sizeof(uint64_t), N,
                                      cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        kmer_b200_result_free(res);
        return fail(KMER_B200_ERR_CUDA, std::string("search_routed: ") + cudaGetErrorString(e));
    }
    *out = res;
    return KMER_B200_OK;
}

int kmer_b200_unroute_device(kmer_b200_index *ix, uint8_t *d_send_blocks, uint8_t *d_ret_blocks, const kmer_b200_route_plan *plan,
                             const uint32_t *sent_counts, const uint32_t *d_recv_positions, const uint64_t *recv_splits, uint64_t Q,
                             const uint8_t *d_status, kmer_b200_result **out) {
    KB_TRY(routable(ix));
    if (!plan || !d_send_blocks || !d_ret_blocks || !sent_counts || !recv_splits || !out || (Q && !d_status))
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    cudaStream_t st = ix->stream;
    const uint32_t N = plan->n_parts;
    kb::RoutePrefix sent{};
    kb::RoutePrefix64 seg{};
    for (uint32_t b = 0; b < N; ++b) {
        sent.p[b + 1] = sent.p[b] + sent_counts[b];
        seg.p[b + 1] = seg.p[b] + recv_splits[b];
    }
    kmer_b200_result *res = device_result_new(ix, Q);
    if (!res) return KMER_B200_ERR_OUT_OF_MEMORY;
    uint64_t *d_block_sums = nullptr;
    auto bail = [&](int code) {
        dev_free(ix, d_block_sums);
        kmer_b200_result_free(res);
        return code;
    };
    if (dev_alloc(ix, &d_block_sums, kb::offsets_scan_blocks(Q) + 1, false)) return bail(KMER_B200_ERR_OUT_OF_MEMORY);
    cudaMemsetAsync(res->offsets, 0, (Q + 1) * sizeof(uint64_t), st);
    if (Q) cudaMemcpyAsync(res->status, d_status, Q, cudaMemcpyDeviceToDevice, st);
    kb::launch_unroute_counts(d_send_blocks, plan->block_bytes, plan->stride, d_ret_blocks, plan->return_block_bytes, plan->capacity, N, sent,
                              res->offsets, res->status, st);
    kb::launch_offsets_scan(res->offsets, Q, d_block_sums, st);
    uint64_t total = 0;
    cudaError_t e = cudaMemcpyAsync(&total, res->offsets + Q, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return bail(fail(KMER_B200_ERR_CUDA, std::string("unroute: ") + cudaGetErrorString(e)));
    if (total != seg.p[N]) return bail(fail(KMER_B200_ERR_INVALID_ARGUMENT, "unroute: the return blocks and the received positions disagree"));
    res->n_positions = total;
    if (total) {
        if (!d_recv_positions) return bail(fail(KMER_B200_ERR_INVALID_ARGUMENT, "null positions"));
        if (dev_alloc(ix, &res->positions, total, false)) return bail(KMER_B200_ERR_OUT_OF_MEMORY);
        kb::launch_unroute_place(d_send_blocks, plan->block_bytes, plan->stride, d_ret_blocks, plan->return_block_bytes, plan->capacity, N, sent,
                                 seg, d_recv_positions, res->offsets, res->positions, st);
    }
    dev_free(ix, d_block_sums);
    d_block_sums = nullptr;
    e = cudaGetLastError();
    if (e != cudaSuccess) return bail(fail(KMER_B200_ERR_CUDA, std::string("unroute: ") + cudaGetErrorString(e)));
    *out = res;
    return KMER_B200_OK;
}

uint64_t kmer_b200_presence_words(const kmer_b200_index *ix, uint32_t e) {
    ix = primary(ix);
    if (!ix || e >= ix->ks.size()) return 0;
    return (ix->elems[e].dev.key_space + 63) / 64 + 1;
}

int kmer_b200_presence_export(kmer_b200_index *ix, uint32_t e, uint64_t *d_bitmap) {
    if (!ix || !d_bitmap || e >= ix->ks.size() || !ix->replicas.empty()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    KB_TRY(reject_view(ix, e));
    const HostElement &he = ix->elems[e];
    if (he.dev.shift != 0) return fail(KMER_B200_ERR_UNSUPPORTED, "presence bitmaps come from dense directories");
    DeviceGuard guard(ix->device);
    const uint64_t lo = he.dev.key_lo, hi = he.dev.key_hi == UINT64_MAX ? he.dev.key_space : he.dev.key_hi;
    if (lo % 64) return fail(KMER_B200_ERR_UNSUPPORTED, "part boundary not on a 64-hash boundary");
    kb::launch_presence_bits(he.d_dir, hi - lo, d_bitmap + lo / 64, ix->stream);
    KB_CUDA(cudaGetLastError());
    return KMER_B200_OK;
}

int kmer_b200_presence_attach(kmer_b200_index *ix, uint32_t e, const uint64_t *d_bitmap) {
    if (!ix || e >= ix->ks.size() || !ix->replicas.empty()) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    KB_TRY(reject_view(ix, e));
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    ix->host_index.presence[e] = d_bitmap;  // caller-owned; null detaches
    KB_CUDA(cudaMemcpyAsync(ix->d_index, &ix->host_index, sizeof(kb::DeviceIndex), cudaMemcpyHostToDevice, ix->stream));
    KB_CUDA(cudaStreamSynchronize(ix->stream));
    return KMER_B200_OK;
}

// ---- several devices behind one handle (kmer_b200_config.n_devices > 1) ----------------------------------------------
// Build: one host thread per device builds that device's key-range part from the host text (its own H2D over its own
// PCIe link, 1 / N of the sorting work); then every part is pushed to every other device with peer copies, so all
// devices end up with the whole index. Indices that cannot be cut into key-range parts (64-bit hashes) are simply built
// whole on every device.
static int create_multi(const uint8_t *ranks, uint64_t n, uint32_t sigma, const uint32_t *ks, uint32_t n_ks,
                        const kmer_b200_config *cfg_in, kmer_b200_index **out, const uint8_t *lut256) {
    if (!out) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "out is null");
    *out = nullptr;
    const uint32_t N = cfg_in->n_devices;
    if (!cfg_in->device_ids || N > 64) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "device_ids is null or n_devices > 64");
    if (cfg_in->n_total || cfg_in->shard_begin || cfg_in->halo || cfg_in->key_parts > 1 || cfg_in->stream)
        return fail(KMER_B200_ERR_INVALID_ARGUMENT, "a multi-device index takes the whole text and its own streams");
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) {
        cudaGetLastError();
        return fail(KMER_B200_ERR_CUDA, "no usable CUDA device (libkmer_b200 has no CPU fallback)");
    }
    std::vector<int> ids(cfg_in->device_ids, cfg_in->device_ids + N);
    for (uint32_t i = 0; i < N; ++i) {
        if (ids[i] < 0 || ids[i] >= count) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "device id out of range");
        for (uint32_t j = 0; j < i; ++j)
            if (ids[j] == ids[i]) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "duplicate device id");
    }
    bool pool_shared = true;  // every device may read the other devices' pool allocations from a kernel
    {
        DeviceGuard keep(ids[0]);
        for (uint32_t i = 0; i < N; ++i) {
            cudaSetDevice(ids[i]);
            for (uint32_t j = 0; j < N; ++j)
                if (j != i) cudaDeviceEnablePeerAccess(ids[j], 0);  // direct NVLink copies; staged through the host otherwise
            cudaGetLastError();
            // the library allocates from the device's stream-ordered pool, which peer access does not cover by itself:
            // kernels on the other devices read this device's position part
            cudaMemPool_t pool;
            if (cudaDeviceGetDefaultMemPool(&pool, ids[i]) == cudaSuccess) {
                std::vector<cudaMemAccessDesc> acc;
                for (uint32_t j = 0; j < N; ++j) {
                    if (j == i) continue;
                    cudaMemAccessDesc d{};
                    d.location.type = cudaMemLocationTypeDevice;
                    d.location.id = ids[j];
                    d.flags = cudaMemAccessFlagsProtReadWrite;
                    acc.push_back(d);
                }
                if (!acc.empty() && cudaMemPoolSetAccess(pool, acc.data(), acc.size()) != cudaSuccess) pool_shared = false;
            } else {
                pool_shared = false;
            }
            cudaGetLastError();
        }
    }
    std::vector<kmer_b200_index *> reps(N, nullptr);
    std::vector<int> rc(N, 0);
    std::vector<std::string> err(N);
    auto build_all = [&](uint32_t parts) {
        std::vector<std::thread> th;
        for (uint32_t i = 0; i < N; ++i)
            th.emplace_back([&, i] {
                kmer_b200_config c = *cfg_in;
                c.device = ids[i];
                c.n_devices = 0;
                c.device_ids = nullptr;
                c.key_part = parts > 1 ? i : 0;
                c.key_parts = parts > 1 ? parts : 0;
                c.reserved |= kFlagPlainTextUpload;
                rc[i] = create_impl(ranks, false, n, sigma, ks, n_ks, &c, &reps[i], lut256);
                if (rc[i] != 0) err[i] = g_last_error;
            });
        for (auto &t : th) t.join();
    };
    auto destroy_all = [&] {
        for (auto &r : reps) {
            kmer_b200_destroy(r);
            r = nullptr;
        }
    };
    build_all(N);
    bool parts = true;
    for (uint32_t i = 0; i < N; ++i)
        if (rc[i] == KMER_B200_ERR_UNSUPPORTED) parts = false;
    if (!parts) {  // no key-range parts for this index: every device builds the whole of it
        destroy_all();
        build_all(1);
    }
    for (uint32_t i = 0; i < N; ++i)
        if (rc[i] != 0) {
            const int code = rc[i];
            const std::string msg = err[i];
            destroy_all();
            return fail(code, msg);
        }
    auto bail = [&](int code, const std::string &msg) {
        destroy_all();
        return fail(code, msg);
    };
    for (uint32_t e = 0; parts && e < n_ks; ++e) {
        const uint64_t n_kmers = n - ks[e] + 1;
        const uint64_t key_space = reps[0]->elems[e].dev.key_space;
        std::vector<uint64_t> base(N + 1, 0);
        for (uint32_t i = 0; i < N; ++i) base[i + 1] = base[i] + reps[i]->elems[e].dev.n_kmers;
        if (base[N] != n_kmers) return bail(KMER_B200_ERR_CUDA, "multi-device build: the parts do not add up to the whole index");
        // Preferred assembly (up to 8 devices, no bucket beyond 254 entries, equal key ranges): the positions stay where
        // they were sorted -- every device reads the other devices' parts over NVLink (peer access, same process) -- and
        // only the directory is made whole everywhere, shipped as one byte per bucket and prefix-summed on arrival.
        if (N <= (uint32_t)kb::kMaxPosParts && pool_shared) {
            std::vector<uint8_t *> sizes(N, nullptr), sizes_full(N, nullptr);
            std::vector<uint32_t *> dir_whole(N, nullptr);
            auto drop = [&] {
                for (uint32_t d = 0; d < N; ++d) {
                    DeviceGuard g(ids[d]);
                    dev_free(reps[d], sizes[d]);
                    dev_free(reps[d], sizes_full[d]);
                    sizes[d] = sizes_full[d] = nullptr;
                }
            };
            bool ok = true;
            uint64_t width0 = reps[0]->elems[e].dev.key_hi - reps[0]->elems[e].dev.key_lo;
            for (uint32_t i = 0; ok && i < N; ++i) {
                DeviceGuard g(ids[i]);
                const HostElement &he = reps[i]->elems[e];
                const uint64_t w = he.dev.key_hi - he.dev.key_lo;
                ok = he.dev.shift == 0 && he.dev.key_lo == (uint64_t)i * width0 && (w == width0 || i + 1 == N);
                uint64_t n_large = 0;
                if (ok) ok = dev_alloc(reps[i], &sizes[i], std::max<uint64_t>(w, 1), false) == 0 &&
                             kmer_b200_export_bucket_sizes(reps[i], e, sizes[i], &n_large) == 0 && n_large == 0;
            }
            for (uint32_t d = 0; ok && d < N; ++d) {
                DeviceGuard g(ids[d]);
                ok = dev_alloc(reps[d], &sizes_full[d], key_space, false) == 0 && dev_alloc(reps[d], &dir_whole[d], key_space + 1, false) == 0;
                if (ok) ok = cudaStreamSynchronize(reps[d]->stream) == cudaSuccess;  // the allocations exist before peers write them
            }
            for (uint32_t i = 0; ok && i < N; ++i) {
                DeviceGuard g(ids[i]);
                const HostElement &he = reps[i]->elems[e];
                const uint64_t w = he.dev.key_hi - he.dev.key_lo;
                for (uint32_t d = 0; w && d < N; ++d)
                    cudaMemcpyPeerAsync(sizes_full[d] + he.dev.key_lo, ids[d], sizes[i], ids[i], w, reps[i]->stream);
            }
            for (uint32_t i = 0; ok && i < N; ++i) {
                DeviceGuard g(ids[i]);
                ok = cudaStreamSynchronize(reps[i]->stream) == cudaSuccess && cudaGetLastError() == cudaSuccess;
            }
            for (uint32_t d = 0; ok && d < N; ++d) {
                DeviceGuard g(ids[d]);
                ok = kmer_b200_directory_from_sizes(reps[d], sizes_full[d], key_space, dir_whole[d]) == 0;
            }
            if (ok) {
                std::vector<const uint32_t *> part_ptrs(N);
                for (uint32_t i = 0; i < N; ++i) part_ptrs[i] = reps[i]->elems[e].d_pos;
                for (uint32_t d = 0; ok && d < N; ++d) {
                    DeviceGuard g(ids[d]);
                    ok = cudaStreamSynchronize(reps[d]->stream) == cudaSuccess &&
                         adopt_parts_impl(reps[d], e, part_ptrs.data(), base.data(), N, dir_whole[d], key_space + 1, true) == 0;
                    if (ok) dir_whole[d] = nullptr;  // the index owns it now
                }
                if (!ok) {
                    drop();
                    return bail(KMER_B200_ERR_CUDA, "multi-device build: adopting the parts failed: " + g_last_error);
                }
                drop();
                continue;
            }
            cudaGetLastError();
            drop();
            for (uint32_t d = 0; d < N; ++d) {
                DeviceGuard g(ids[d]);
                dev_free(reps[d], dir_whole[d]);
            }
        }
        std::vector<uint32_t *> pos_full(N, nullptr), dir_full(N, nullptr);
        for (uint32_t d = 0; d < N; ++d) {
            DeviceGuard g(ids[d]);
            if (dev_alloc(reps[d], &pos_full[d], n_kmers, false) || dev_alloc(reps[d], &dir_full[d], key_space + 1, false))
                return bail(KMER_B200_ERR_OUT_OF_MEMORY, g_last_error);
        }
        // every device: its own part into its own whole arrays (positions copied, directory offset by the earlier parts)
        std::vector<uint64_t> lo(N), n_dir(N);
        for (uint32_t i = 0; i < N; ++i) {
            DeviceGuard g(ids[i]);
            const HostElement &he = reps[i]->elems[e];
            lo[i] = he.dev.key_lo;
            n_dir[i] = he.dev.key_hi - he.dev.key_lo + (i + 1 == N ? 1 : 0);
            const uint64_t cnt = he.dev.n_kmers;
            if (cnt) cudaMemcpyAsync(pos_full[i] + base[i], he.d_pos, cnt * 4, cudaMemcpyDeviceToDevice, reps[i]->stream);
            if (n_dir[i])
                add_base32_kernel<<<(unsigned)((n_dir[i] + 255) / 256), 256, 0, reps[i]->stream>>>(he.d_dir, n_dir[i], (uint32_t)base[i],
                                                                                                  dir_full[i] + lo[i]);
        }
        for (uint32_t i = 0; i < N; ++i) {
            DeviceGuard g(ids[i]);
            if (cudaStreamSynchronize(reps[i]->stream) != cudaSuccess) return bail(KMER_B200_ERR_CUDA, "multi-device build: part export failed");
        }
        // ... and pushed to every other device (NVLink peer copies, all sources at once)
        for (uint32_t i = 0; i < N; ++i) {
            DeviceGuard g(ids[i]);
            const uint64_t cnt = base[i + 1] - base[i];
            for (uint32_t d = 0; d < N; ++d) {
                if (d == i) continue;
                if (cnt) cudaMemcpyPeerAsync(pos_full[d] + base[i], ids[d], pos_full[i] + base[i], ids[i], cnt * 4, reps[i]->stream);
                if (n_dir[i]) cudaMemcpyPeerAsync(dir_full[d] + lo[i], ids[d], dir_full[i] + lo[i], ids[i], n_dir[i] * 4, reps[i]->stream);
            }
        }
        for (uint32_t i = 0; i < N; ++i) {
            DeviceGuard g(ids[i]);
            if (cudaStreamSynchronize(reps[i]->stream) != cudaSuccess || cudaGetLastError() != cudaSuccess)
                return bail(KMER_B200_ERR_CUDA, "multi-device build: peer copy failed");
        }
        for (uint32_t d = 0; d < N; ++d) {
            const int s = adopt_element_impl(reps[d], e, pos_full[d], n_kmers, dir_full[d], key_space + 1, 2);
            if (s != 0) return bail(s, g_last_error);
        }
    }
    kmer_b200_index *group = new (std::nothrow) kmer_b200_index();
    if (!group) return bail(KMER_B200_ERR_OUT_OF_MEMORY, "host allocation failed");
    group->device = ids[0];
    for (kmer_b200_index *r : reps) r->host_sharers = N;
    group->cfg = *cfg_in;
    group->cfg.device_ids = nullptr;
    group->n = n;
    group->sigma = sigma;
    group->bits = reps[0]->bits;
    group->ks.assign(ks, ks + n_ks);
    group->replicas = reps;
    *out = group;
    return KMER_B200_OK;
}

// A host batch on a multi-device handle: device i takes the queries [Q i / N, Q (i + 1) / N) -- its own upload, search
// and download, all devices at once -- and the slices are concatenated into one result.
static int search_batch_multi(kmer_b200_index *group, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t Q, uint32_t mode,
                              const uint8_t *lut256, kmer_b200_result **out) {
    const uint32_t N = (uint32_t)group->replicas.size();
    std::vector<kmer_b200_result *> part(N, nullptr);
    std::vector<int> rc(N, 0);
    std::vector<std::string> err(N);
    std::vector<uint64_t> q0(N + 1);
    for (uint32_t i = 0; i <= N; ++i) q0[i] = Q * i / N;
    {
        std::vector<std::thread> th;
        for (uint32_t i = 0; i < N; ++i)
            th.emplace_back([&, i] {
                rc[i] = search_batch_host(group->replicas[i], q_ranks, q_offsets + q0[i], q0[i + 1] - q0[i], mode, lut256, &part[i]);
                if (rc[i] != 0) err[i] = g_last_error;
            });
        for (auto &t : th) t.join();
    }
    auto free_parts = [&] {
        for (auto *r : part) kmer_b200_result_free(r);
    };
    for (uint32_t i = 0; i < N; ++i)
        if (rc[i] != 0) {
            const int code = rc[i];
            const std::string msg = err[i];
            free_parts();
            return fail(code, msg);
        }
    std::vector<uint64_t> p0(N + 1, 0);
    for (uint32_t i = 0; i < N; ++i) p0[i + 1] = p0[i] + part[i]->n_positions;
    kmer_b200_result *res = host_result_new(group, Q);
    if (!res || !host_result_positions(res, p0[N])) {
        free_parts();
        kmer_b200_result_free(res);
        return fail(KMER_B200_ERR_OUT_OF_MEMORY, "host allocation failed");
    }
    {
        std::vector<std::thread> th;
        for (uint32_t i = 0; i < N; ++i)
            th.emplace_back([&, i] {
                const uint64_t Qi = q0[i + 1] - q0[i];
                const uint64_t *so = part[i]->offsets;
                uint64_t *dof = res->offsets + q0[i];
                for (uint64_t j = 0; j < Qi; ++j) dof[j] = so[j] + p0[i];
                if (Qi) std::memcpy(res->status + q0[i], part[i]->status, Qi);
                if (part[i]->n_positions) std::memcpy(res->positions + p0[i], part[i]->positions, part[i]->n_positions * sizeof(uint32_t));
            });
        for (auto &t : th) t.join();
    }
    res->offsets[Q] = p0[N];
    free_parts();
    *out = res;
    return KMER_B200_OK;
}

uint64_t kmer_b200_scheme(const kmer_b200_index *ix, uint64_t m, uint32_t *out_ks, uint64_t cap, int *use_multi) {
    ix = primary(ix);
    if (!ix || m >= kb::kQuerySizeRange) return 0;
    const uint32_t o = ix->sum_off[m], len = ix->sum_off[m + 1] - o;
    for (uint32_t i = 0; i < len && i < cap && out_ks; ++i) out_ks[i] = ix->ks[ix->sum_elem[o + i]];
    if (use_multi) *use_multi = ix->use_multi[m];
    return len;
}

static int element_occupancy(kmer_b200_index *ix, HostElement &he) {
    if (he.n_occupied || he.dev.n_kmers == 0) return 0;
    unsigned long long *d_cnt = nullptr;
    KB_TRY(dev_alloc(ix, &d_cnt, 1, false));
    cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), ix->stream);
    const unsigned grid = kb::device_sm_count() * 16;
    if (he.dev.shift == 0)
        count_steps_kernel<<<grid, 256, 0, ix->stream>>>(he.d_dir, he.dev.dir_entries - 1, d_cnt);
    else if (he.key_bytes == 8)
        count_steps_kernel<<<grid, 256, 0, ix->stream>>>((const uint64_t *)he.d_keys, he.dev.n_kmers - 1, d_cnt);
    else
        count_steps_kernel<<<grid, 256, 0, ix->stream>>>((const uint32_t *)he.d_keys, he.dev.n_kmers - 1, d_cnt);
    unsigned long long c = 0;
    KB_CUDA(cudaMemcpyAsync(&c, d_cnt, sizeof(c), cudaMemcpyDeviceToHost, ix->stream));
    KB_CUDA(cudaStreamSynchronize(ix->stream));
    dev_free(ix, d_cnt);
    he.n_occupied = he.dev.shift == 0 ? c : c + 1;  // run starts = steps + 1
    return 0;
}

int kmer_b200_plan_table(kmer_b200_index *ix, uint32_t mode, uint32_t m_lo, uint32_t m_hi, kmer_b200_plan_row *out) {
    ix = primary(ix);
    if (!ix || !out || m_lo == 0 || m_hi < m_lo) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad argument");
    if (ix->cfg.reserved & KMER_B200_FLAG_SHARED_POSITIONS)
        return fail(KMER_B200_ERR_UNSUPPORTED, "plan table: bucket statistics are per element; build the index without shared positions");
    if (mode == UINT32_MAX) mode = ix->cfg.mode;
    DeviceGuard guard(ix->device);
    std::lock_guard<std::mutex> lock(ix->mu);
    const uint32_t n_ks = (uint32_t)ix->ks.size();
    for (uint32_t e = 0; e < n_ks; ++e) KB_TRY(element_occupancy(ix, ix->elems[e]));
    auto mean_bucket = [&](uint32_t e) {
        const HostElement &he = ix->elems[e];
        return he.n_occupied ? (double)he.dev.n_kmers / (double)he.n_occupied : 0.0;
    };
    auto largest_k_at_most = [&](uint32_t m, uint32_t *e_out) {  // element with the largest k <= m
        bool found = false;
        for (uint32_t e = 0; e < n_ks; ++e)
            if (ix->ks[e] <= m && (!found || ix->ks[e] > ix->ks[*e_out])) {
                *e_out = e;
                found = true;
            }
        return found;
    };
    const double sym_per_sector = 256.0 / ix->bits;
    for (uint32_t m = m_lo; m <= m_hi; ++m) {
        kmer_b200_plan_row &r = out[m - m_lo];
        r = kmer_b200_plan_row{};
        r.m = m;
        uint32_t e0 = 0, k0 = 0;
        bool throws = false, defective = false, multi_sum = false, sub_k = false;
        uint32_t n_lookups = 1;
        if (mode == KMER_B200_MODE_CORRECT) {
            // the smallest k >= m (bucket or prefix slab = the result, nothing to verify), else the largest k
            bool found = false;
            for (uint32_t e = 0; e < n_ks; ++e)
                if (ix->ks[e] >= m && (!found || ix->ks[e] < ix->ks[e0])) {
                    e0 = e;
                    found = true;
                }
            if (!found) largest_k_at_most(m, &e0);
            k0 = ix->ks[e0];
            sub_k = k0 > m;
        } else {
            if (m >= kb::kQuerySizeRange) {
                r.kind = 5;
                continue;
            }
            const uint32_t so = ix->sum_off[m], sl = ix->sum_off[m + 1] - so;
            e0 = ix->sum_elem[so];
            k0 = ix->ks[e0];
            const bool multi = ix->use_multi[m] && n_ks > 1;
            if (!multi) {
                if (m < k0) {
                    sub_k = true;
                    throws = std::pow((double)ix->sigma, (double)(k0 - m)) > 1e7;  // kmer_index.hpp:119-122
                } else if (m > k0) {
                    const uint32_t P = m / k0, rest = m % k0;
                    const bool throw_after = rest > 0 && std::pow((double)ix->sigma, (double)(k0 - rest)) > 1e7;
                    defective = rest != 0 && P > 2;
                    if (throw_after) throws = true;  // once every full part occurs somewhere
                    if (throw_after || defective) n_lookups = P;
                }
            } else if (sl >= 3) {
                multi_sum = true;
                n_lookups = sl;
            }
            // contiguous plans give the same occurrences from any element: the largest k <= m has the shortest buckets
            if (!sub_k && !defective && !multi_sum) {
                uint32_t e = e0;
                if (largest_k_at_most(m, &e)) e0 = e, k0 = ix->ks[e];
            }
        }
        r.seed_k = k0;
        r.n_lookups = n_lookups;
        if (throws && (sub_k || n_lookups == 1)) {
            r.kind = 5;
            r.expected_sectors = n_lookups;
            continue;
        }
        if (sub_k) {
            r.kind = 1;
            r.expected_candidates = (double)ix->elems[e0].dev.n_kmers / std::pow((double)ix->sigma, (double)m);
            r.n_lookups = 2;
            r.expected_sectors = 2 + r.expected_candidates / 8.0;
            continue;
        }
        r.kind = throws ? 5 : (m == k0 ? 0 : (defective ? 3 : (multi_sum ? 4 : 2)));
        r.expected_candidates = mean_bucket(e0);
        const double verify = m == k0 ? 0.0 : 1.0 + std::floor((double)m / sym_per_sector);
        r.expected_sectors = n_lookups * (ix->elems[e0].dev.shift ? 2.0 : 1.0) + std::ceil(r.expected_candidates / 8.0) +
                             r.expected_candidates * verify;
    }
    return KMER_B200_OK;
}

uint64_t kmer_b200_scheme_for_ks(const uint32_t *ks, uint32_t n_ks, uint64_t m, uint32_t *out_ks, uint64_t cap,
                                 int *use_multi) {
    if (!ks || n_ks == 0 || n_ks > (uint32_t)kb::kMaxElements || m >= kb::kQuerySizeRange) return 0;
    for (uint32_t i = 0; i < n_ks; ++i)
        if (ks[i] == 0 || ks[i] > 63) return 0;
    // the table only depends on the ks; cache the last one built (tests walk m for a fixed ks)
    static std::mutex mu;
    static SchemeHost cached;
    std::lock_guard<std::mutex> lock(mu);
    if (cached.ks != std::vector<uint32_t>(ks, ks + n_ks)) {
        cached = SchemeHost();
        cached.ks.assign(ks, ks + n_ks);
        build_scheme(&cached);
    }
    const uint32_t o = cached.sum_off[m], len = cached.sum_off[m + 1] - o;
    for (uint32_t i = 0; i < len && i < cap && out_ks; ++i) out_ks[i] = cached.ks[cached.sum_elem[o + i]];
    if (use_multi) *use_multi = cached.use_multi[m];
    return len;
}

uint32_t kmer_b200_stats(kmer_b200_index *ix, kmer_b200_kernel_stat *out, uint32_t cap) {
    ix = primary(ix);  // a multi-device handle reports its first device
    if (!ix) return 0;
    DeviceGuard guard(ix->device);
    ix->prof.resolve();
    uint32_t n = 0;
    for (int i = 0; i < K_COUNT_ && n < cap; ++i) {
        if (out) {
            out[n].name = kKernelNames[i];
            out[n].launches = ix->prof.launches[i];
            out[n].device_ms = ix->prof.ms[i];
            out[n].algorithmic_bytes = ix->prof.bytes[i];
        }
        ++n;
    }
    return n;
}

void kmer_b200_stats_reset(kmer_b200_index *ix) {
    if (!ix) return;
    if (!ix->replicas.empty()) {
        for (kmer_b200_index *r : ix->replicas) kmer_b200_stats_reset(r);
        return;
    }
    DeviceGuard guard(ix->device);
    ix->prof.reset();
}

uint64_t kmer_b200_device_bytes(const kmer_b200_index *ix) {
    if (!ix) return 0;
    uint64_t total = ix->device_bytes;
    for (const kmer_b200_index *r : ix->replicas) total += r->device_bytes;  // all devices of a multi-device handle
    return total;
}

uint64_t kmer_b200_debug_guard_violations(void) {
    if (!guard_mode() || !g_guard_bad) return 0;
    int n_dev = 0, prev = 0;
    cudaGetDeviceCount(&n_dev);
    cudaGetDevice(&prev);
    for (int d = 0; d < n_dev; ++d) {  // the checks run on the streams the buffers were freed on
        cudaSetDevice(d);
        cudaDeviceSynchronize();
    }
    cudaSetDevice(prev);
    cudaGetLastError();
    return *reinterpret_cast<volatile unsigned long long *>(g_guard_bad);
}

int kmer_b200_debug_guard_selftest(void) {
    // one allocation, one store a byte behind its end, one a byte before its start: both must be counted
    if (!guard_mode()) return fail(KMER_B200_ERR_UNSUPPORTED, "KMER_B200_GUARD is not set");
    const uint64_t before = kmer_b200_debug_guard_violations();
    uint8_t *p = nullptr;
    KB_CUDA(kb_malloc_async((void **)&p, 1000, nullptr));
    KB_CUDA(cudaMemsetAsync(p + 1000, 0, 1, nullptr));
    KB_CUDA(cudaMemsetAsync(p - 1, 0, 1, nullptr));
    kb_free_async(p, nullptr);
    return kmer_b200_debug_guard_violations() - before == 2 ? KMER_B200_OK
                                                             : fail(KMER_B200_ERR_CUDA, "guard zones did not see the stores");
}

uint64_t kmer_b200_last_search_gathers(const kmer_b200_index *ix) { return ix ? primary(ix)->last_gathers : 0; }

uint64_t kmer_b200_build_transfer(const kmer_b200_index *ix) {
    if (!ix) return 0;
    if (ix->replicas.empty()) return ix->build_h2d;
    uint64_t sum = 0;
    for (const kmer_b200_index *r : ix->replicas) sum += r->build_h2d;
    return sum;
}

void kmer_b200_last_search_host_path(const kmer_b200_index *ix, uint32_t *pipeline, uint32_t *raw_pct, double *pack_gbs) {
    const kmer_b200_index *p = ix && !ix->replicas.empty() ? ix->replicas[0] : ix;
    if (pipeline) *pipeline = p ? p->last_host_path : 0;
    if (raw_pct) *raw_pct = p ? p->last_raw_pct : 0;
    if (pack_gbs) *pack_gbs = p ? p->last_pack_gbs : 0;
}

uint64_t kmer_b200_host_pack_stream_words(uint64_t n, uint32_t sigma) {
    return kb::pack_stream_words(n, sigma <= 4 ? 2 : (sigma <= 16 ? 4 : 8));
}

int kmer_b200_host_pack_stream(const uint8_t *ranks, uint64_t n, uint32_t sigma, uint64_t *words) {
    if ((n && !ranks) || !words || sigma < 2 || sigma > 256) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null argument or sigma out of range");
    const uint32_t bits = sigma <= 4 ? 2 : (sigma <= 16 ? 4 : 8);
    kb::HostPool &pool = kb::HostPool::instance();
    const unsigned parts = std::max(1u, std::min(pool.threads() * 4, 256u));
    std::vector<uint8_t> ok(parts, 1);
    pool.run(parts, [&](unsigned t) { ok[t] = kb::pack_stream_host(ranks, n, bits, sigma, words, t, parts) ? 1 : 0; });
    for (uint8_t v : ok)
        if (!v) return fail(KMER_B200_ERR_INVALID_RANK, "a rank is >= sigma");
    return KMER_B200_OK;
}

void kmer_b200_last_search_transfer(const kmer_b200_index *ix, uint64_t *h2d_bytes, uint64_t *d2h_bytes) {
    uint64_t in = 0, back = 0;
    if (ix && !ix->replicas.empty()) {
        for (const kmer_b200_index *r : ix->replicas) in += r->last_h2d, back += r->last_d2h;
    } else if (ix) {
        in = ix->last_h2d, back = ix->last_d2h;
    }
    if (h2d_bytes) *h2d_bytes = in;
    if (d2h_bytes) *d2h_bytes = back;
}

int kmer_b200_gather_probe(uint64_t table_bytes, uint64_t n_gathers, void *stream, double *ms_out) {
    if (!ms_out || table_bytes < 4096 || n_gathers == 0) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad probe arguments");
    cudaStream_t st = (cudaStream_t)stream;
    uint64_t *table = nullptr, *sink = nullptr;
    const uint64_t n_words = table_bytes / 8;
    KB_CUDA(cudaMalloc((void **)&table, n_words * 8));
    KB_CUDA(cudaMalloc((void **)&sink, 8));
    KB_CUDA(cudaMemsetAsync(table, 1, n_words * 8, st));
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    kb::launch_gather_probe(table, n_words, std::min<uint64_t>(n_gathers, 1u << 24), sink, st);  // warm-up
    cudaEventRecord(a, st);
    kb::launch_gather_probe(table, n_words, n_gathers, sink, st);
    cudaEventRecord(b, st);
    cudaError_t e = cudaEventSynchronize(b);
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(table);
    cudaFree(sink);
    if (e != cudaSuccess) return fail(KMER_B200_ERR_CUDA, cudaGetErrorString(e));
    *ms_out = ms;
    return KMER_B200_OK;
}

int kmer_b200_gather_probe_at(const void *d_table, uint64_t table_bytes, uint64_t n_gathers, void *stream, double *ms_out) {
    if (!ms_out || !d_table || table_bytes < 4096 || n_gathers == 0) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "bad probe arguments");
    cudaStream_t st = (cudaStream_t)stream;
    uint64_t *sink = nullptr;
    const uint64_t n_words = table_bytes / 8;
    KB_CUDA(cudaMalloc((void **)&sink, 8));
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    kb::launch_gather_probe((const uint64_t *)d_table, n_words, std::min<uint64_t>(n_gathers, 1u << 24), sink, st);  // warm-up
    cudaEventRecord(a, st);
    kb::launch_gather_probe((const uint64_t *)d_table, n_words, n_gathers, sink, st);
    cudaEventRecord(b, st);
    cudaError_t e = cudaEventSynchronize(b);
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(sink);
    if (e != cudaSuccess) return fail(KMER_B200_ERR_CUDA, cudaGetErrorString(e));
    *ms_out = ms;
    return KMER_B200_OK;
}

uint64_t kmer_b200_fast_pow(uint64_t base, uint8_t exp) { return fast_pow(base, exp); }

uint64_t kmer_b200_hash(const uint8_t *ranks, uint32_t k, uint32_t sigma) {
    uint64_t h = 0;
    for (uint32_t i = 0; i < k; ++i) h += (uint64_t)ranks[i] * fast_pow(sigma, (uint8_t)(k - i - 1));
    return h;
}

uint64_t kmer_b200_choose_best_k(const uint64_t *lens, uint64_t n_lens, uint64_t n_k, uint64_t *out_ks) {
    // choose_best_k.hpp:12-60. Candidates in the reference's priority order; the first candidate that divides
    // the length (+3) or misses a multiple by at most 3 (+4 - miss) takes the length's points.
    static const uint64_t cand[10] = {29, 27, 25, 23, 21, 19, 17, 13, 11, 10};
    uint64_t score[10] = {};
    for (uint64_t a = 0; a < n_lens; ++a)
        for (int c = 0; c < 10; ++c) {
            const uint64_t rem = lens[a] % cand[c];
            if (rem == 0) {
                score[c] += 3;
                break;
            }
            if (cand[c] - rem <= 3) {
                score[c] += 4 - (cand[c] - rem);
                break;
            }
        }
    int order[10] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9};
    std::stable_sort(order, order + 10, [&](int x, int y) { return score[x] > score[y]; });
    uint64_t w = 0;
    for (; w < n_k && w < 10; ++w) out_ks[w] = cand[order[w]];
    return w;
}

int kmer_b200_synth_ranks_device(uint8_t *d_out, uint64_t n, uint64_t start, uint32_t sigma, uint64_t seed, void *stream) {
    if (!d_out && n) return fail(KMER_B200_ERR_INVALID_ARGUMENT, "null output");
    kb::launch_synth_ranks(d_out, n, start, sigma, seed, (cudaStream_t)stream);
    KB_CUDA(cudaGetLastError());
    return KMER_B200_OK;
}

}  // extern "C"
