// k-mer spectrum of one index element (sm_100a): the occurrence count of every hash h is its bucket size, so the
// histogram of counts, the number of distinct k-mers and the most frequent k-mers are read off the directory (and the
// sorted hashes of a sparse directory) without touching the positions.
//
// Counts come from one of three sources (SpectrumArgs::source):
//   dense  (shift 0): count(h) = dir[h + 1] - dir[h] for h < sigma^k. spectrum_dense_kernel streams the directory with
//          16-byte loads, 16 entries per thread and round plus the first entry of the next chunk;
//   runs   (shift > 0): a bucket is a run of equal sorted hashes, and a run never crosses a directory block
//          [dir[j], dir[j + 1]): a run start ends at the upper bound of its hash inside its block;
//   slabs  (a view of a shared-positions index, Element::width != 1): count(h) is the owner's slab
//          [h * width, (h + 1) * width), two lower_bound_key per hash (one carried over from the previous hash).
//
// Accumulation: counts 1 and 2 (on a random text nearly every non-empty bucket) are counted in registers and summed per
// warp once, at the end; counts below kSpecSmemBins go to a per-CTA shared-memory histogram, larger ones straight to the
// global one; every CTA flushes once. An empty bucket costs its load.
//
// Corrections (a small open-addressing table of (hash, delta)): on a collection index every window that crosses a record
// start is charged to the first start above it (delta -1), on a view every tail start of the text (no owner k-mer starts
// there) gets delta +1. spectrum_correct_kernel then moves each affected hash from its raw bin to its corrected one.
//
// Selection (frequent list, exact cutoff): every hash whose corrected count is >= a threshold, in hash order, by a count
// pass (per-tile totals), launch_offsets_scan and a write pass; the host sorts the selection by count.
#include "launch.h"

namespace kb {

namespace {

constexpr int kSpecThreads = 256;
constexpr uint32_t kSpecSmemBins = 4096;  // bins held in shared memory (16 KB); larger counts go to global atomics
constexpr uint32_t kDenseChunk = 16;      // directory entries per thread and round of the dense sweep
constexpr uint32_t kTileItems = 8;        // items per thread of the generic sweeps
constexpr uint64_t kTile = (uint64_t)kSpecThreads * kTileItems;
constexpr uint64_t kNoKey = ~0ull;        // an empty table slot (no hash reaches 2^64 - 1: sigma^k < 2^64)
constexpr uint32_t kFull = 0xFFFFFFFFu;

__device__ __forceinline__ uint64_t warp_sum64(uint64_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ uint64_t warp_max64(uint64_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, (uint64_t)__shfl_xor_sync(kFull, v, o));
    return v;
}

__device__ __forceinline__ uint64_t table_slot(uint64_t h, uint32_t mask) {
    h ^= h >> 33;
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    return h & mask;
}

__device__ __forceinline__ void table_add(const SpectrumArgs &s, uint64_t h, int delta) {
    for (uint64_t i = table_slot(h, s.tab_mask);; i = (i + 1) & s.tab_mask) {
        const unsigned long long prev = atomicCAS(&s.tab_keys[i], kNoKey, (unsigned long long)h);
        if (prev == kNoKey || prev == h) {
            atomicAdd(&s.tab_delta[i], delta);
            return;
        }
    }
}

__device__ __forceinline__ int table_get(const SpectrumArgs &s, uint64_t h) {
    for (uint64_t i = table_slot(h, s.tab_mask);; i = (i + 1) & s.tab_mask) {
        const unsigned long long key = s.tab_keys[i];
        if (key == h) return s.tab_delta[i];
        if (key == kNoKey) return 0;
    }
}

struct SpecAcc {
    uint32_t n1 = 0, n2 = 0;
    uint64_t distinct = 0, max = 0;

    __device__ __forceinline__ void add(uint64_t c, uint32_t *sh, uint32_t sh_bins, const SpectrumArgs &s) {
        if (c == 0) return;
        ++distinct;
        max = c > max ? c : max;
        if (c == 1) {
            ++n1;
        } else if (c == 2) {
            ++n2;
        } else {
            const uint64_t b = min(c, (uint64_t)s.n_bins - 1);
            if (b < sh_bins)
                atomicAdd(&sh[b], 1u);
            else
                atomicAdd(&s.hist[b], 1ull);
        }
    }

    // every thread of the CTA calls once
    __device__ __forceinline__ void flush(uint32_t *sh, uint32_t sh_bins, const SpectrumArgs &s) {
        const uint32_t w1 = __reduce_add_sync(kFull, n1), w2 = __reduce_add_sync(kFull, n2);
        const uint64_t wd = warp_sum64(distinct), wm = warp_max64(max);
        if ((threadIdx.x & 31) == 0) {
            if (w1) atomicAdd(&sh[min(1u, s.n_bins - 1)], w1);
            if (w2) atomicAdd(&sh[min(2u, s.n_bins - 1)], w2);
            if (wd) atomicAdd(&s.stats[0], (unsigned long long)wd);
            if (wm) atomicMax(&s.stats[1], (unsigned long long)wm);
        }
        __syncthreads();
        for (uint32_t b = threadIdx.x; b < sh_bins; b += blockDim.x)
            if (sh[b]) atomicAdd(&s.hist[b], (unsigned long long)sh[b]);
    }
};

__device__ __forceinline__ uint32_t smem_bins_init(uint32_t *sh, const SpectrumArgs &s) {
    const uint32_t sh_bins = min(s.n_bins, kSpecSmemBins);
    for (uint32_t b = threadIdx.x; b < sh_bins; b += blockDim.x) sh[b] = 0;
    __syncthreads();
    return sh_bins;
}

__device__ __forceinline__ uint4 load_stream(const uint32_t *p) {
    uint4 v;
    asm("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

// the hot path: one read of the sigma^k + 1 directory entries
__global__ void __launch_bounds__(kSpecThreads) spectrum_dense_kernel(const SpectrumArgs s) {
    __shared__ uint32_t sh[kSpecSmemBins];
    const uint32_t sh_bins = smem_bins_init(sh, s);
    const uint32_t *__restrict__ dir = s.E.dir;
    const uint64_t n_chunks = s.n_items / kDenseChunk;
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (uint64_t)gridDim.x * blockDim.x;
    SpecAcc a;
    for (uint64_t c = tid; c < n_chunks; c += stride) {
        const uint32_t *p = dir + c * kDenseChunk;
        uint32_t w[kDenseChunk + 1];
#pragma unroll
        for (uint32_t u = 0; u < kDenseChunk / 4; ++u) {
            const uint4 v = load_stream(p + 4 * u);
            w[4 * u] = v.x;
            w[4 * u + 1] = v.y;
            w[4 * u + 2] = v.z;
            w[4 * u + 3] = v.w;
        }
        w[kDenseChunk] = __ldg(p + kDenseChunk);  // the next chunk's first entry (a neighbouring lane streams it)
#pragma unroll
        for (uint32_t j = 0; j < kDenseChunk; ++j) a.add(w[j + 1] - w[j], sh, sh_bins, s);
    }
    const uint64_t t = n_chunks * kDenseChunk + tid;  // the last sigma^k mod 16 buckets
    if (t < s.n_items) a.add(dir[t + 1] - dir[t], sh, sh_bins, s);
    a.flush(sh, sh_bins, s);
}

// f(h, count) for every bucket among the items [i0, i1) of the source (dense: hashes; runs: sorted hashes, one call per
// run start; slabs: hashes of the view's k)
template <int SRC, typename F>
__device__ __forceinline__ void walk(const SpectrumArgs &s, uint64_t i0, uint64_t i1, F &&f) {
    const Element &E = s.E;
    if (SRC == kSpectrumDense) {
        uint32_t lo = E.dir[i0];
        for (uint64_t i = i0; i < i1; ++i) {
            const uint32_t hi = E.dir[i + 1];
            f(i, (uint64_t)(hi - lo));
            lo = hi;
        }
    } else if (SRC == kSpectrumSlabs) {
        uint64_t lo = lower_bound_key(E, i0 * E.width);
        for (uint64_t i = i0; i < i1; ++i) {
            const uint64_t hi = lower_bound_key(E, (i + 1) * E.width);
            f(i, hi - lo);
            lo = hi;
        }
    } else {
        uint64_t prev = i0 ? element_key(E, i0 - 1) : 0;
        for (uint64_t i = i0; i < i1; ++i) {
            const uint64_t key = element_key(E, i);
            if (i == 0 || key != prev) {
                uint64_t a = i + 1, b = gather32(E.dir + (key >> E.shift) + 1);  // the run ends inside its block
                while (a < b) {
                    const uint64_t mid = a + ((b - a) >> 1);
                    if (element_key(E, mid) <= key)
                        a = mid + 1;
                    else
                        b = mid;
                }
                f(key, a - i);
            }
            prev = key;
        }
    }
}

template <int SRC>
__global__ void __launch_bounds__(kSpecThreads) spectrum_sweep_kernel(const SpectrumArgs s) {
    __shared__ uint32_t sh[kSpecSmemBins];
    const uint32_t sh_bins = smem_bins_init(sh, s);
    SpecAcc a;
    const uint64_t n_tiles = (s.n_items + kTile - 1) / kTile;
    for (uint64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint64_t i0 = tile * kTile + (uint64_t)threadIdx.x * kTileItems;
        const uint64_t i1 = min(i0 + kTileItems, s.n_items);
        if (i0 < i1) walk<SRC>(s, i0, i1, [&](uint64_t, uint64_t c) { a.add(c, sh, sh_bins, s); });
    }
    a.flush(sh, sh_bins, s);
}

// corrections: junction r in [1, R) (windows charged to record start r, delta -1) and tail t (delta +1)
__global__ void __launch_bounds__(kSpecThreads) spectrum_corrections_kernel(const SpectrumArgs s, PackedText T, const uint64_t *starts,
                                                                            uint64_t n_records, uint32_t n_tail) {
    const uint32_t k = s.E.k;
    const uint64_t n_junctions = n_records ? n_records - 1 : 0;
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_junctions + n_tail; w += (uint64_t)gridDim.x * blockDim.x) {
        if (w < n_junctions) {
            // windows p < s < p + k with no start in (p, s): p in [max(s - k + 1, previous start), min(s - 1, n - k)]
            const uint64_t st = starts[w + 1], prev = starts[w];
            if (st == 0 || st <= prev) continue;
            const uint64_t lo = max(st + 1 >= k ? st + 1 - k : 0, prev);
            const uint64_t hi = min(st - 1, T.n - k);
            for (uint64_t p = lo; p <= hi; ++p) table_add(s, key_at(T.words, p, k, T.bits, T.sigma), -1);
        } else {
            const uint64_t p = T.n - s.E.k_phys + 1 + (w - n_junctions);
            table_add(s, key_at(T.words, p, k, T.bits, T.sigma), 1);
        }
    }
}

__global__ void __launch_bounds__(kSpecThreads) spectrum_correct_kernel(const SpectrumArgs s) {
    const uint64_t cap = (uint64_t)s.tab_mask + 1;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t h = s.tab_keys[i];
        const int d = s.tab_delta[i];
        if (h == kNoKey || d == 0) continue;
        const uint64_t raw = bucket_of<true>(s.E, h).cnt, c = (uint64_t)((int64_t)raw + d);
        const uint64_t last = s.n_bins - 1;
        if (raw) {
            atomicAdd(&s.hist[min(raw, last)], ~0ull);  // - 1
            atomicAdd(&s.stats[0], ~0ull);
        }
        if (c) {
            atomicAdd(&s.hist[min(c, last)], 1ull);
            atomicAdd(&s.stats[0], 1ull);
        }
        atomicAdd(&s.stats[2], (unsigned long long)(int64_t)d);
    }
}

// one CTA per tile of kTile items: count pass -> sel.tile[tile] = selected hashes (and stats[3] = their largest count);
// write pass (sel.tile = exclusive offsets) -> hashes and counts in hash order
template <int SRC>
__global__ void __launch_bounds__(kSpecThreads) spectrum_select_kernel(const SpectrumArgs s, const SpectrumSelect sel, bool write) {
    __shared__ uint32_t warp_n[kSpecThreads / 32];
    const uint64_t tile = blockIdx.x;
    const uint64_t i0 = tile * kTile + (uint64_t)threadIdx.x * kTileItems;
    const uint64_t i1 = min(i0 + kTileItems, s.n_items);
    const bool has_table = s.tab_keys != nullptr;
    auto corrected = [&](uint64_t h, uint64_t raw) -> uint64_t {
        // deltas are <= 0 on a collection: a raw count below the threshold stays below it
        if (has_table && (s.tail || raw >= sel.thr)) return (uint64_t)((int64_t)raw + table_get(s, h));
        return raw;
    };
    uint32_t n = 0;
    uint64_t mx = 0;
    if (i0 < i1)
        walk<SRC>(s, i0, i1, [&](uint64_t h, uint64_t raw) {
            const uint64_t c = corrected(h, raw);
            if (c >= sel.thr) {
                ++n;
                mx = max(mx, c);
            }
        });
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) warp_n[warp] = incl;
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kSpecThreads / 32; ++w) {
        before += w < warp ? warp_n[w] : 0;
        total += warp_n[w];
    }
    if (!write) {
        mx = warp_max64(mx);
        if (lane == 0 && mx) atomicMax(&s.stats[3], (unsigned long long)mx);
        if (threadIdx.x == 0) sel.tile[tile] = total;
        return;
    }
    if (n == 0) return;
    uint64_t o = sel.tile[tile] + before + incl - n;
    walk<SRC>(s, i0, i1, [&](uint64_t h, uint64_t raw) {
        const uint64_t c = corrected(h, raw);
        if (c >= sel.thr) {
            sel.hashes[o] = h;
            sel.counts[o] = (uint32_t)c;
            ++o;
        }
    });
}

// sort input: key = max_count - count (ascending = count descending), value = selection index
__global__ void __launch_bounds__(kSpecThreads) spectrum_sort_keys_kernel(const uint32_t *counts, uint64_t n, uint32_t max_count,
                                                                          uint32_t *keys, uint32_t *vals) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        keys[i] = max_count - counts[i];
        vals[i] = (uint32_t)i;
    }
}

__global__ void __launch_bounds__(kSpecThreads) spectrum_gather_kernel(const uint64_t *hashes, const uint32_t *counts, const uint32_t *order,
                                                                       uint64_t n, uint64_t *out_hashes, uint64_t *out_counts) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t j = order ? order[i] : (uint32_t)i;
        out_hashes[i] = hashes[j];
        out_counts[i] = counts[j];
    }
}

// one CTA per resident slot: a grid-stride sweep with more CTAs than fit at once ends in a partial wave
template <typename K>
unsigned resident_grid(K kernel) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kSpecThreads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    return device_sm_count() * (unsigned)per_sm;
}

unsigned grid_for(uint64_t n) {
    return (unsigned)std::min<uint64_t>((n + kSpecThreads - 1) / kSpecThreads, (uint64_t)device_sm_count() * 8);
}

}  // namespace

uint64_t spectrum_tiles(uint64_t n_items) { return (n_items + kTile - 1) / kTile; }

void launch_spectrum_sweep(const SpectrumArgs &s, cudaStream_t stream) {
    if (s.n_items == 0) return;
    const uint64_t tiles = spectrum_tiles(s.n_items);
    auto sweep = [&](auto kernel) { kernel<<<(unsigned)std::min<uint64_t>(tiles, resident_grid(kernel)), kSpecThreads, 0, stream>>>(s); };
    switch (s.source) {
        case kSpectrumDense:
            // 16-byte loads need a 16-byte aligned directory (always so for the library's; an adopted one may not be)
            if (((uintptr_t)s.E.dir & 15) == 0)
                spectrum_dense_kernel<<<resident_grid(spectrum_dense_kernel), kSpecThreads, 0, stream>>>(s);
            else
                sweep(spectrum_sweep_kernel<kSpectrumDense>);
            break;
        case kSpectrumRuns: sweep(spectrum_sweep_kernel<kSpectrumRuns>); break;
        default: sweep(spectrum_sweep_kernel<kSpectrumSlabs>); break;
    }
}

void launch_spectrum_corrections(const SpectrumArgs &s, const PackedText &text, const uint64_t *d_starts, uint64_t n_records,
                                 uint32_t n_tail, cudaStream_t stream) {
    const uint64_t work = (n_records ? n_records - 1 : 0) + n_tail;
    if (work == 0) return;
    spectrum_corrections_kernel<<<grid_for(work), kSpecThreads, 0, stream>>>(s, text, d_starts, n_records, n_tail);
    spectrum_correct_kernel<<<grid_for((uint64_t)s.tab_mask + 1), kSpecThreads, 0, stream>>>(s);
}

void launch_spectrum_select(const SpectrumArgs &s, const SpectrumSelect &sel, bool write, cudaStream_t stream) {
    const uint64_t tiles = spectrum_tiles(s.n_items);
    if (tiles == 0) return;
    switch (s.source) {
        case kSpectrumDense: spectrum_select_kernel<kSpectrumDense><<<(unsigned)tiles, kSpecThreads, 0, stream>>>(s, sel, write); break;
        case kSpectrumRuns: spectrum_select_kernel<kSpectrumRuns><<<(unsigned)tiles, kSpecThreads, 0, stream>>>(s, sel, write); break;
        default: spectrum_select_kernel<kSpectrumSlabs><<<(unsigned)tiles, kSpecThreads, 0, stream>>>(s, sel, write); break;
    }
}

void launch_spectrum_sort_keys(const uint32_t *d_counts, uint64_t n, uint32_t max_count, uint32_t *d_keys, uint32_t *d_vals,
                               cudaStream_t stream) {
    if (n) spectrum_sort_keys_kernel<<<grid_for(n), kSpecThreads, 0, stream>>>(d_counts, n, max_count, d_keys, d_vals);
}

void launch_spectrum_gather(const uint64_t *d_hashes, const uint32_t *d_counts, const uint32_t *d_order, uint64_t n, uint64_t *d_out_hashes,
                            uint64_t *d_out_counts, cudaStream_t stream) {
    if (n) spectrum_gather_kernel<<<grid_for(n), kSpecThreads, 0, stream>>>(d_hashes, d_counts, d_order, n, d_out_hashes, d_out_counts);
}

}  // namespace kb
