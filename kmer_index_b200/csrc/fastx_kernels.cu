// FASTA / FASTQ bytes -> ranks on the device (SURVEY.md 8f.3: the step in front of the path -- the reference's callers
// assign characters to alphabet objects one by one before the index ever sees them, test_main.cpp:13-17,
// benchmarks/input_generator.hpp:52-63). The file is parsed where it lands in HBM: header lines, line breaks (and, for
// FASTQ, the '+' and quality lines) are dropped, sequence characters go through a 256-entry rank table, the records
// are concatenated into ONE text and a record table (start of every record in that text, byte offset of its header
// line) is produced, so that hit positions map back to (record, offset).
//
// Three passes over tiles of 2048 bytes: (1) per tile: number of line feeds, position of the last one; a small scan
// carries "which line am I in / where did it start" across tiles; (2) per tile: kept symbols and record starts ->
// exclusive scans; (3) the same classification again, now writing ranks and record starts at their final places.
#include "launch.h"

namespace kb {

constexpr int kFxThreads = 256;
constexpr int kFxPer = 8;
constexpr int kFxTile = kFxThreads * kFxPer;  // 2048 bytes

__device__ __forceinline__ int64_t block_scan_max_excl(int64_t v, int64_t *warp_buf) {
    // exclusive max-scan over the block's threads (identity = -1)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl = max(incl, t);
    }
    if (lane == 31) warp_buf[warp] = incl;
    __syncthreads();
    int64_t before = -1;
    for (int w = 0; w < warp; ++w) before = max(before, warp_buf[w]);
    int64_t excl = __shfl_up_sync(0xFFFFFFFFu, incl, 1);
    if (lane == 0) excl = -1;
    __syncthreads();
    return max(before, excl);
}

__device__ __forceinline__ uint32_t block_scan_sum_excl(uint32_t v, uint32_t *warp_buf, uint32_t *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_buf[warp] = incl;
    __syncthreads();
    uint32_t before = 0, all = 0;
    for (int w = 0; w < kFxThreads / 32; ++w) {
        if (w < warp) before += warp_buf[w];
        all += warp_buf[w];
    }
    __syncthreads();
    if (total) *total = all;
    return before + incl - v;
}

// pass 1: line feeds per tile, global position of the tile's last line feed (-1: none)
__global__ void __launch_bounds__(kFxThreads) fastx_tile_stats_kernel(const uint8_t *__restrict__ data, uint64_t n, uint64_t *__restrict__ nl_count,
                                                                       int64_t *__restrict__ last_nl) {
    __shared__ uint32_t s_cnt;
    __shared__ long long s_last;
    if (threadIdx.x == 0) {
        s_cnt = 0;
        s_last = -1;
    }
    __syncthreads();
    const uint64_t i0 = (uint64_t)blockIdx.x * kFxTile + (uint64_t)threadIdx.x * kFxPer;
    uint32_t c = 0;
    long long last = -1;
    for (int j = 0; j < kFxPer; ++j)
        if (i0 + j < n && data[i0 + j] == '\n') {
            ++c;
            last = (long long)(i0 + j);
        }
    if (c) {
        atomicAdd(&s_cnt, c);
        atomicMax(&s_last, last);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        nl_count[blockIdx.x] = s_cnt;
        last_nl[blockIdx.x] = s_last;
    }
}

// carry across tiles (single CTA): last_nl[t] <- position of the last line feed BEFORE tile t (-1: none)
__global__ void __launch_bounds__(1024) fastx_carry_kernel(int64_t *__restrict__ last_nl, uint64_t n_tiles) {
    __shared__ int64_t part[1024];
    const uint64_t per = (n_tiles + 1023) / 1024;
    const uint64_t t0 = (uint64_t)threadIdx.x * per, t1 = min(t0 + per, n_tiles);
    int64_t mx = -1;
    for (uint64_t t = t0; t < t1; ++t) mx = max(mx, last_nl[t]);
    part[threadIdx.x] = mx;
    __syncthreads();
    int64_t run = -1;
    for (int i = 0; i < (int)threadIdx.x; ++i) run = max(run, part[i]);
    for (uint64_t t = t0; t < t1; ++t) {
        const int64_t v = last_nl[t];
        last_nl[t] = run;
        run = max(run, v);
    }
}

struct FxClass {
    bool keep[kFxPer];       // a sequence symbol
    bool rec_start[kFxPer];  // first byte of a record's header line
};

// classification of the thread's kFxPer bytes. format 1 = FASTA (header lines start with '>' or ';'), 2 = FASTQ (records of
// four lines: @name, sequence, +, qualities; an empty line where a header would be starts no record)
__device__ __forceinline__ FxClass fastx_classify(const uint8_t *__restrict__ data, uint64_t n, uint32_t format, uint64_t nl_before_tile,
                                                  int64_t last_nl_before_tile, int64_t *warp_buf64, uint32_t *warp_buf32, uint8_t (&ch)[kFxPer]) {
    const uint64_t i0 = (uint64_t)blockIdx.x * kFxTile + (uint64_t)threadIdx.x * kFxPer;
    uint32_t nl_mine = 0;
    int64_t last_mine = -1;
    for (int j = 0; j < kFxPer; ++j) {
        ch[j] = i0 + j < n ? data[i0 + j] : (uint8_t)'\n';
        if (i0 + j < n && ch[j] == '\n') {
            ++nl_mine;
            last_mine = (int64_t)(i0 + j);
        }
    }
    const int64_t last_before = max(last_nl_before_tile, block_scan_max_excl(last_mine, warp_buf64));  // last line feed before my first byte
    const uint64_t nl_before = nl_before_tile + block_scan_sum_excl(nl_mine, warp_buf32, nullptr);
    FxClass c;
    int64_t line_start = last_before + 1;
    uint64_t line_no = nl_before;
    for (int j = 0; j < kFxPer; ++j) {
        const uint64_t i = i0 + j;
        c.keep[j] = false;
        c.rec_start[j] = false;
        if (i < n) {
            const uint8_t first = (uint64_t)line_start == i ? ch[j] : data[line_start];  // first byte of this byte's line
            bool header, seq_line;
            if (format == 2) {
                // an empty line in header position is no record (a file that ends in a blank line); a blank line
                // between records moves the next '@' line to a sequence line, where '@' is refused
                header = (line_no & 3) == 0 && first != '\n' && first != '\r';
                seq_line = (line_no & 3) == 1;
            } else {
                header = first == '>' || first == ';';
                seq_line = !header;
            }
            c.rec_start[j] = header && (uint64_t)line_start == i && !(format != 2 && first == ';');
            c.keep[j] = seq_line && ch[j] != '\n' && ch[j] != '\r' && ch[j] != ' ' && ch[j] != '\t';
            if (ch[j] == '\n') {
                line_start = (int64_t)i + 1;
                ++line_no;
            }
        }
    }
    return c;
}

// pass 2: kept symbols and record starts per tile
__global__ void __launch_bounds__(kFxThreads) fastx_count_kernel(const uint8_t *__restrict__ data, uint64_t n, uint32_t format,
                                                                  const uint64_t *__restrict__ nl_before, const int64_t *__restrict__ last_nl,
                                                                  uint64_t *__restrict__ kept, uint64_t *__restrict__ recs) {
    __shared__ int64_t wb64[kFxThreads / 32];
    __shared__ uint32_t wb32[kFxThreads / 32];
    uint8_t ch[kFxPer];
    const FxClass c = fastx_classify(data, n, format, nl_before[blockIdx.x], last_nl[blockIdx.x], wb64, wb32, ch);
    uint32_t k = 0, r = 0;
    for (int j = 0; j < kFxPer; ++j) {
        k += c.keep[j];
        r += c.rec_start[j];
    }
    uint32_t tk = 0, tr = 0;
    block_scan_sum_excl(k, wb32, &tk);
    block_scan_sum_excl(r, wb32, &tr);
    if (threadIdx.x == 0) {
        kept[blockIdx.x] = tk;
        recs[blockIdx.x] = tr;
    }
}

// pass 3: ranks and record table
__global__ void __launch_bounds__(kFxThreads) fastx_write_kernel(const uint8_t *__restrict__ data, uint64_t n, uint32_t format,
                                                                  const uint64_t *__restrict__ nl_before, const int64_t *__restrict__ last_nl,
                                                                  const uint64_t *__restrict__ kept_off, const uint64_t *__restrict__ recs_off,
                                                                  const uint8_t *__restrict__ lut, uint32_t sigma, uint8_t *__restrict__ ranks,
                                                                  uint64_t *__restrict__ rec_start_symbol, uint64_t *__restrict__ rec_header_byte,
                                                                  uint32_t *__restrict__ error_flag) {
    __shared__ int64_t wb64[kFxThreads / 32];
    __shared__ uint32_t wb32[kFxThreads / 32];
    __shared__ uint8_t s_lut[256];
    s_lut[threadIdx.x] = lut[threadIdx.x];
    uint8_t ch[kFxPer];
    const FxClass c = fastx_classify(data, n, format, nl_before[blockIdx.x], last_nl[blockIdx.x], wb64, wb32, ch);
    uint32_t k = 0, r = 0;
    for (int j = 0; j < kFxPer; ++j) {
        k += c.keep[j];
        r += c.rec_start[j];
    }
    uint64_t ko = kept_off[blockIdx.x] + block_scan_sum_excl(k, wb32, nullptr);
    uint64_t ro = recs_off[blockIdx.x] + block_scan_sum_excl(r, wb32, nullptr);
    const uint64_t i0 = (uint64_t)blockIdx.x * kFxTile + (uint64_t)threadIdx.x * kFxPer;
    bool bad = false;
    for (int j = 0; j < kFxPer; ++j) {
        if (c.rec_start[j]) {
            rec_start_symbol[ro] = ko;  // the record's sequence starts at the next kept symbol
            rec_header_byte[ro] = i0 + j;
            ++ro;
        }
        if (c.keep[j]) {
            const uint8_t rk = s_lut[ch[j]];
            bad |= rk >= sigma;
            ranks[ko++] = rk;
        }
    }
    if (bad) atomicOr(error_flag, 1u);
}

uint64_t fastx_tiles(uint64_t n_bytes) { return (n_bytes + kFxTile - 1) / kFxTile; }

void launch_fastx_tile_stats(const uint8_t *d_data, uint64_t n, uint64_t *d_nl_count, int64_t *d_last_nl, cudaStream_t stream) {
    fastx_tile_stats_kernel<<<(unsigned)fastx_tiles(n), kFxThreads, 0, stream>>>(d_data, n, d_nl_count, d_last_nl);
    fastx_carry_kernel<<<1, 1024, 0, stream>>>(d_last_nl, fastx_tiles(n));
}
void launch_fastx_count(const uint8_t *d_data, uint64_t n, uint32_t format, const uint64_t *d_nl_before, const int64_t *d_last_nl,
                        uint64_t *d_kept, uint64_t *d_recs, cudaStream_t stream) {
    fastx_count_kernel<<<(unsigned)fastx_tiles(n), kFxThreads, 0, stream>>>(d_data, n, format, d_nl_before, d_last_nl, d_kept, d_recs);
}
void launch_fastx_write(const uint8_t *d_data, uint64_t n, uint32_t format, const uint64_t *d_nl_before, const int64_t *d_last_nl,
                        const uint64_t *d_kept_off, const uint64_t *d_recs_off, const uint8_t *d_lut, uint32_t sigma, uint8_t *d_ranks,
                        uint64_t *d_rec_start_symbol, uint64_t *d_rec_header_byte, uint32_t *d_error_flag, cudaStream_t stream) {
    fastx_write_kernel<<<(unsigned)fastx_tiles(n), kFxThreads, 0, stream>>>(d_data, n, format, d_nl_before, d_last_nl, d_kept_off, d_recs_off,
                                                                            d_lut, sigma, d_ranks, d_rec_start_symbol, d_rec_header_byte,
                                                                            d_error_flag);
}

}  // namespace kb
