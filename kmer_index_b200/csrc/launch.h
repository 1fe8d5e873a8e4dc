// Host-callable launchers of the kernels in build_kernels.cu / search_kernels.cu / synth.cu.
#pragma once

#include "common.cuh"

namespace kb {

// ---- build
void launch_pack_text(const uint8_t *d_ranks, uint64_t n, uint32_t bits, uint32_t sigma, uint64_t n_words_total,
                      uint64_t *d_words, uint32_t *d_error_flag, cudaStream_t stream);
void launch_hist_text(const PackedText &text, uint32_t k, uint64_t n_kmers, uint32_t shift, uint32_t mask,
                      uint32_t *d_tile_hist, cudaStream_t stream);
void launch_hist_pairs(const void *d_keys, uint32_t key_bytes, uint64_t n, uint32_t shift, uint32_t mask,
                       uint32_t *d_tile_hist, cudaStream_t stream);
void launch_column_scan(uint32_t *d_tile_hist, uint32_t n_tiles, uint32_t *d_chunk_sums, cudaStream_t stream);
// key_bytes: 4 (sigma^k <= 2^32) or 8
void launch_scatter_text(const PackedText &text, uint32_t k, uint32_t key_bytes, uint64_t n_kmers, uint32_t shift,
                         uint32_t mask, const uint32_t *d_tile_base, void *d_out_keys, uint32_t *d_out_vals,
                         cudaStream_t stream);
void launch_scatter_pairs(const void *d_keys, const uint32_t *d_vals, uint32_t key_bytes, uint64_t n, uint32_t shift,
                          uint32_t mask, const uint32_t *d_tile_base, void *d_out_keys, uint32_t *d_out_vals,
                          cudaStream_t stream);
void launch_directory_fill(const void *d_keys, uint32_t key_bytes, uint64_t n_kmers, uint32_t shift, uint64_t dir_entries,
                           uint32_t *d_dir, cudaStream_t stream);
uint32_t sort_tile_size();
uint32_t scan_chunk_tiles();
// ---- single-sweep sorter for 32-bit hashes (onesweep.cu)
// global digit histograms of every pass -> d_digit_base[p][256] (exclusive prefixes); d_hist_scratch: 8 * 256 u32.
// from_cmers: power-of-two alphabet with w_bits a multiple of the symbol width (one c-mer histogram serves all passes)
void launch_digit_histograms(const PackedText &text, uint32_t k, uint64_t n_kmers, uint32_t n_passes, uint32_t w_bits,
                             uint32_t key_bits, bool from_cmers, uint32_t *d_hist_scratch, uint32_t *d_digit_base,
                             cudaStream_t stream);
// one scatter pass. text != null: pass 0 (hashes from the packed text, positions generated); else pairs in.
// d_out_pairs == null: final pass, writes d_out_vals (+ d_out_keys when non-null). d_status: zeroed u64[n_tiles][256]
// shared by the passes of one sort (tag = pass + 1); d_tile_counter: one zeroed u32 per pass.
void launch_onesweep_pass(const PackedText *text, uint32_t k, const uint2 *d_in_pairs, uint64_t n, uint32_t shift, uint32_t mask,
                          uint32_t tag, const uint32_t *d_digit_base, uint64_t *d_status, uint32_t *d_tile_counter,
                          uint2 *d_out_pairs, uint32_t *d_out_keys, uint32_t *d_out_vals, cudaStream_t stream);
uint32_t device_sm_count();
// key-range parts: (hash - lo, position) pairs of the k-mers with hash in [lo, hi), in position order.
// count -> launch_offsets_scan over the u64 tile counts -> write
uint32_t filter_tiles(uint64_t n_kmers);
void launch_owned_count(const PackedText &text, uint32_t k, uint64_t n_kmers, uint64_t lo, uint64_t hi, uint64_t *d_tile_counts,
                        cudaStream_t stream);
void launch_owned_write(const PackedText &text, uint32_t k, uint64_t n_kmers, uint64_t lo, uint64_t hi, const uint64_t *d_tile_offsets,
                        uint32_t *d_out_keys, uint32_t *d_out_vals, cudaStream_t stream);
void launch_digit_histograms_pairs(const uint2 *d_pairs, uint64_t n, uint32_t n_passes, uint32_t w_bits, uint32_t *d_hist_scratch,
                                   uint32_t *d_digit_base, cudaStream_t stream);

// ---- search
enum SearchPass : int {
    kPassCount = 0,
    kPassWrite = 1,
    kPassPresence = 2,
    kPassCountAccount = 3,   // count + gather accounting
    kPassCountDeferred = 4,  // sharded: count + per-part presence flags, whole-text rule applied afterwards
    kPassCountDeferredAccount = 5
};

struct SearchArgs {
    const DeviceIndex *index;        // device pointer
    const uint8_t *q_ranks;          // device
    const uint64_t *q_offsets;       // device, [Q + 1]
    // alternative input (q_packed != null; q_ranks / q_offsets unused): queries already packed like the text, b bits
    // per symbol MSB-first, query i in words [i * q_stride, (i + 1) * q_stride), its length in q_lens16[i]; ranks were
    // validated by the packer (host threads of kmer_b200_search_batch)
    const uint64_t *q_packed;
    const uint16_t *q_lens16;
    uint32_t q_stride;
    uint64_t n_queries;
    uint32_t mode;                   // kmer_b200_mode
    uint32_t group;                  // lanes per query: 1, 2, 4, 8 or 32
    uint32_t bits;                   // bits per packed symbol (to size the heavy launch's staging)
    uint32_t single_k;               // the index has one element: launch the kernels compiled without the multi-k plans
    uint32_t lean_ok;                // host-checked: single k, dna4 (2-bit symbols), dense 32-bit directory, plain count pass ->
                                     // search_lean.cu may take the count pass when max_len <= 128
    struct {                         // Element::n_pos_parts / part_first / pos_part of element 0 (peer-positions index)
        uint32_t n;
        uint32_t first[kMaxPosParts + 1];
        const uint32_t *ptr[kMaxPosParts];
    } parts0;
    uint32_t views;                  // shared-positions index (Element::width != 1 exists): the warp-per-query kernels compiled
                                     // with view support run every pass
    uint32_t *heavy;                 // device or null, u32[1 + Q]: [0] = number of heavy queries, then their ids
    uint32_t *hits;                  // device or null, u32[1 + Q]: [0] = number of queries with hits (count pass), then their ids
    uint32_t q_words;                // packed words reserved per query in shared memory (search_q_words)
    uint32_t max_len;                // longest query the shared-memory reservation (and the shard halo) allows
    const uint64_t *present_global;  // device or null: OR over shards of the presence masks (format 0)
    const uint32_t *present_global4; // device or null: SUM over shards of the nibble-encoded masks (format 1)
    uint32_t *present4;              // device (presence pass, format 1), [Q]: bit 4j = part j occurs in this shard
    uint64_t *counts;                // device, [Q + 1]: per-query hit counts (count pass), then offsets
    uint8_t *status;                 // device, [Q]
    uint8_t *unsorted;               // device, [Q]: 1 = the written segment still needs sorting (sub-k)
    uint32_t *positions;             // device (write pass)
    uint8_t *defer;                  // device (deferred count pass), [Q]: 0x40 | throw << 7 | parts, 0 = no rule applies
    uint64_t *present;               // device (presence pass), [Q]
    unsigned long long *gather_count;  // device or null: accumulates the 32-byte sectors the batch must gather
    uint32_t *error_flag;            // device u32[4]: [0] bit 0 = query rank >= sigma; [1] = #segments to sort;
                                     // [2..3] = u64 mask of sub-k query lengths that found no auxiliary element
    uint32_t approx;                 // 1: approximate search (search_approx.cu): every window within max_mismatches substitutions;
                                     // 2: the same on a collection index (windows inside one record only)
    uint32_t max_mismatches;         // e <= kMaxMismatches
};

// a query with more candidates than this is handed from its group of lanes to the warp-per-query launch
constexpr uint32_t kHeavyCandidates = 2048;

void launch_search(const SearchArgs &args, SearchPass pass, cudaStream_t stream);
// approximate search (search_approx.cu): passes kPassCount, kPassCountAccount and kPassWrite of an unsharded index whose
// elements hold their positions (whole or in peer parts); queries as 1-byte ranks (q_packed unused)
constexpr uint32_t kMaxMismatches = 8;
void launch_search_approx(const SearchArgs &args, SearchPass pass, cudaStream_t stream);
// hit strategies of approximate search (search_approx.cu). kApproxBest: count passes over every query with budget
// min(e, m - 1) -> best_dist / best_pos per query, counts = 1 where a hit exists, those queries listed in args.hits,
// budget[q] = min(e, d_min + strata) when budget != null. kApproxListed: count and write passes over the queries of
// args.hits with budget[q] each (the count pass leaves the list as it is).
enum ApproxMode : int { kApproxAll = 0, kApproxListed = 1, kApproxBest = 2 };
struct ApproxHitArgs {
    uint8_t *budget;     // device or null, [Q]: per-query budget e_q
    uint8_t *best_dist;  // device (kApproxBest), [Q]: d_min, 0xFF = no hit
    uint32_t *best_pos;  // device (kApproxBest), [Q]: the lowest position with d_min
    uint32_t strata;     // s of the strata strategy (0 = all best)
};
void launch_search_approx_hits(const SearchArgs &args, const ApproxHitArgs &h, ApproxMode mode, SearchPass pass,
                               cudaStream_t stream);
// after the offsets scan: positions[offsets[q]] = best_pos[q] (+ distances) for each listed query
void launch_approx_single(const SearchArgs &args, const ApproxHitArgs &h, uint8_t *d_distances, cudaStream_t stream);
// after the write pass (and segment sort): d_distances[j] = d(positions[j]) over the listed queries' hits; budget
// h.budget[q], else args.max_mismatches
void launch_approx_distances(const SearchArgs &args, const ApproxHitArgs &h, uint8_t *d_distances, cudaStream_t stream);
uint32_t search_q_words(uint32_t group, uint32_t bits, uint64_t max_len);
// collection index (search_approx.cu; SearchArgs::approx = 2 selects the record-boundary check of the approximate
// kernels): bit s of d_bits (zeroed, n / 64 + 1 words) = a record starts at s, 0 < s < n; and (record, offset) per position
void launch_record_boundaries(const uint64_t *d_starts, uint64_t n_records, uint64_t n, uint64_t *d_bits, cudaStream_t stream);
void launch_locate(const uint64_t *d_starts, uint64_t n_records, const uint32_t *d_positions, uint64_t n_pos, uint32_t *d_record,
                   uint32_t *d_offset, cudaStream_t stream);
// ---- k-mer seeding (search_seeds.cu): every k-mer of every query looked up in one element, one warp per query
struct HeavySeed {  // a bucket the write pass hands to the warp-per-bucket launch
    uint64_t out;   // its first output slot
    uint64_t cnt;   // hits to write
    uint32_t lo;    // its first CSR entry
    uint32_t j;     // the k-mer's query offset
};
struct SeedArgs {
    const DeviceIndex *index;        // device pointer
    const uint8_t *q_ranks;          // device
    const uint64_t *q_offsets;       // device, [Q + 1]
    uint64_t n_queries;
    uint32_t elem;                   // the element of k (not an auxiliary one)
    uint32_t k;
    uint32_t max_occ;                // 0 = no cap
    uint32_t coll;                   // collection index: in-record windows only
    const uint64_t *kmer_base;       // device, [Q + 1]: index of each query's first k-mer in the batch's k-mer order
    uint32_t *kmer_counts;           // device, [n_kmers]
    uint32_t *bucket_lo;             // device, [n_kmers], or null (count only): each k-mer's first CSR entry
    uint64_t *counts;                // device, [Q + 1]: hits per query (count pass), then offsets
    uint8_t *status;                 // device, [Q]
    uint32_t *positions;             // device (write pass)
    uint32_t *seed_offsets;          // device (write pass): the j of each position
    HeavySeed *heavy;                // device (write pass) or null: room for every bucket above kHeavyCandidates hits
    unsigned long long *n_heavy;     // device: such buckets (count pass), then the heavy list's length (zeroed before the write pass)
    uint32_t *error_flag;            // device u32: bit 0 = query rank >= sigma
    unsigned long long *gather_count;  // device or null: accumulates the 32-byte sectors gathered
};
// n_kmers[q] = max(0, m_q - k + 1), to be turned into SeedArgs::kmer_base by launch_offsets_scan
void launch_seed_kmers_per_query(const uint64_t *d_q_offsets, uint64_t n_queries, uint32_t k, uint64_t *d_n_kmers, cudaStream_t stream);
void launch_seed_count(const SeedArgs &a, cudaStream_t stream);
// after the offsets scan of the count pass's counts: the write pass and, when a.heavy != null, the heavy launch
void launch_seed_write(const SeedArgs &a, cudaStream_t stream);

// deferred count pass epilogue: zero the counts / set THROW according to the combined presence flags
void launch_finalize_deferred(uint64_t *d_counts, uint8_t *d_status, const uint8_t *d_defer, const uint32_t *d_present4_global,
                              uint64_t n_queries, cudaStream_t stream);
// in place: counts[0..Q) -> exclusive offsets, counts[Q] = total
void launch_offsets_scan(uint64_t *d_counts, uint64_t n_queries, uint64_t *d_block_sums, cudaStream_t stream);
uint64_t offsets_scan_blocks(uint64_t n_queries);
// sort the flagged per-query segments of positions ascending (one CTA per flagged segment)
void launch_segment_sort(uint32_t *d_positions, uint32_t *d_tmp, const uint64_t *d_offsets, const uint8_t *d_unsorted,
                         uint64_t n_queries, uint32_t key_bits, cudaStream_t stream);

// ---- query routing of the key-range multi-GPU search (route_kernels.cu)
constexpr int kMaxParts = 64;
struct RoutePrefix {
    uint32_t p[kMaxParts + 1];  // p[b] = records in the blocks before block b
};
struct RoutePrefix64 {
    uint64_t p[kMaxParts + 1];
};
struct RouteArgs {
    const uint8_t *q_ranks;     // device: this rank's slice of the batch
    const uint64_t *q_offsets;  // device, [Q + 1]
    uint64_t n_queries;
    uint32_t mode, bits, sigma, k;
    uint64_t part_width;        // hashes per index part
    uint32_t n_parts, stride, capacity;
    uint8_t *blocks;            // device: n_parts send blocks (counts zeroed)
    uint64_t block_bytes;
    uint8_t *status;            // device, [Q]: 0xFF = routed (the owner decides), else the status decided here
    uint32_t *flags;            // device u32: bit 0 = rank >= sigma, bit 1 = a query cannot be routed, bit 2 = a block overflowed
};
uint64_t route_block_bytes(uint32_t capacity, uint32_t stride);
uint64_t route_return_block_bytes(uint32_t capacity);
void launch_route_pack(const RouteArgs &a, cudaStream_t stream);
void launch_compact_blocks(uint8_t *d_blocks, uint64_t block_bytes, uint32_t n_parts, uint32_t capacity, uint32_t stride,
                           const RoutePrefix &pfx, uint64_t *d_words, uint16_t *d_lens, cudaStream_t stream);
void launch_pack_return(const uint64_t *d_offsets, const uint8_t *d_status, const RoutePrefix &pfx, uint32_t n_parts, uint8_t *d_ret_blocks,
                        uint64_t ret_bytes, uint32_t capacity, cudaStream_t stream);
void launch_unroute_counts(uint8_t *d_send_blocks, uint64_t block_bytes, uint32_t stride, uint8_t *d_ret_blocks, uint64_t ret_bytes,
                           uint32_t capacity, uint32_t n_parts, const RoutePrefix &sent, uint64_t *d_counts, uint8_t *d_status,
                           cudaStream_t stream);
void launch_unroute_place(uint8_t *d_send_blocks, uint64_t block_bytes, uint32_t stride, uint8_t *d_ret_blocks, uint64_t ret_bytes,
                          uint32_t capacity, uint32_t n_parts, const RoutePrefix &sent, const RoutePrefix64 &seg, const uint32_t *d_recv_pos,
                          const uint64_t *d_offsets, uint32_t *d_positions, cudaStream_t stream);
// bit h - lo of d_bits_at_lo = the part's directory says hash h occurs (n_keys = hi - lo hashes)
void launch_presence_bits(const uint32_t *d_dir, uint64_t n_keys, uint64_t *d_bits_at_lo, cudaStream_t stream);

// ---- FASTA / FASTQ parsing on the device (fastx_kernels.cu)
uint64_t fastx_tiles(uint64_t n_bytes);
// d_nl_count[tiles] (u64): line feeds per tile; d_last_nl[tiles]: position of the last line feed before each tile (-1: none)
void launch_fastx_tile_stats(const uint8_t *d_data, uint64_t n, uint64_t *d_nl_count, int64_t *d_last_nl, cudaStream_t stream);
void launch_fastx_count(const uint8_t *d_data, uint64_t n, uint32_t format, const uint64_t *d_nl_before, const int64_t *d_last_nl,
                        uint64_t *d_kept, uint64_t *d_recs, cudaStream_t stream);
void launch_fastx_write(const uint8_t *d_data, uint64_t n, uint32_t format, const uint64_t *d_nl_before, const int64_t *d_last_nl,
                        const uint64_t *d_kept_off, const uint64_t *d_recs_off, const uint8_t *d_lut, uint32_t sigma, uint8_t *d_ranks,
                        uint64_t *d_rec_start_symbol, uint64_t *d_rec_header_byte, uint32_t *d_error_flag, cudaStream_t stream);

// a directory part as one byte per bucket (its size, 255 = "255 or more": counted in *d_n_large), and back: the whole
// directory as the exclusive prefix sum of all sizes (tile sums -> launch_offsets_scan -> offsets)
void launch_bucket_sizes(const uint32_t *d_dir, uint64_t n_keys, uint8_t *d_sizes, unsigned long long *d_n_large, cudaStream_t stream);
uint64_t sizes_tiles(uint64_t n);
void launch_sizes_tile_sums(const uint8_t *d_sizes, uint64_t n, uint64_t *d_tile_sums, cudaStream_t stream);
void launch_sizes_to_dir(const uint8_t *d_sizes, uint64_t n, const uint64_t *d_tile_off, uint32_t *d_dir, cudaStream_t stream);

// ---- random-gather calibration (the denominator of the search roofline)
void launch_gather_probe(const uint64_t *d_table, uint64_t n_words, uint64_t n_gathers, uint64_t *d_sink, cudaStream_t stream);

// ---- synthetic inputs
void launch_synth_ranks(uint8_t *d_out, uint64_t n, uint64_t start, uint32_t sigma, uint64_t seed, cudaStream_t stream);

}  // namespace kb
