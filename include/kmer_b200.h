/*
 * kmer_b200.h -- C ABI of libkmer_b200.so, the B200 (sm_100a) build + batched-search engine behind the
 * header-only C++ API in include/kmer_index.hpp.
 *
 * The reference (Clemapfel/kmer_index) is header-only C++ with no FFI; the boundary replaced here is the
 * body of its templates. Each entry point names the reference interface it stands in for (file:line into
 * the reference tree). Plain C types only: opaque handles, pointers and sizes. All functions return
 * KMER_B200_OK (0) or a negative kmer_b200_status; kmer_b200_last_error() gives the message of the last
 * failure on the calling thread. There is NO CPU fallback: without a CUDA device every entry point that
 * computes returns KMER_B200_ERR_CUDA.
 */
#ifndef KMER_B200_H
#define KMER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMER_B200_ABI_VERSION 2

typedef enum kmer_b200_status {
    KMER_B200_OK = 0,
    KMER_B200_ERR_INVALID_ARGUMENT = -1, /* null pointer, k out of range, n < k, ... */
    KMER_B200_ERR_CUDA = -2,             /* any CUDA runtime failure (including "no device") */
    KMER_B200_ERR_OUT_OF_MEMORY = -3,
    KMER_B200_ERR_INVALID_RANK = -4,     /* a text/query symbol rank >= sigma */
    KMER_B200_ERR_UNSUPPORTED = -5
} kmer_b200_status;

/* Per-query status, mirroring what the reference's search() does for that query. */
typedef enum kmer_b200_query_status {
    KMER_B200_QUERY_OK = 0,
    /* the reference throws std::invalid_argument: "query size too low for specified k"
       (kmer_index.hpp:119-122) or "query size exceed the maximum size" (kmer_index.hpp:507-509) */
    KMER_B200_QUERY_THROW_INVALID_ARGUMENT = 1,
    /* the reference's behaviour is undefined for this query (empty query: assert kmer_index.hpp:195;
       length == 10000: out-of-bounds table read kmer_index.hpp:512); no hits are reported */
    KMER_B200_QUERY_UNDEFINED = 2,
    /* sharded index only: query longer than the shard's halo allows (see kmer_b200_config.halo) */
    KMER_B200_QUERY_TOO_LONG_FOR_SHARD = 3
} kmer_b200_query_status;

/* Search semantics. REFERENCE_EXACT reproduces kmer_index.hpp:193-346 and :505-558 bit for bit,
   including the two defects documented in DESIGN.md (later parts compared against the last part,
   kmer_index.hpp:314; multi-k offsets not accumulated, kmer_index.hpp:526,535,544) and the throw
   conditions. CORRECT returns the true occurrence set of every query and never throws for short rests. */
typedef enum kmer_b200_mode {
    KMER_B200_MODE_REFERENCE_EXACT = 0,
    KMER_B200_MODE_CORRECT = 1
} kmer_b200_mode;

/* kmer_b200_config::reserved */
enum {
    /* never build auxiliary k' = m elements for sub-k query lengths (saves memory; those results are then sorted by the
       segment-sort kernel instead) */
    KMER_B200_FLAG_NO_AUX = 1,
    /* Shared-positions multi-k index (the reference's own outlook, thesis/content/04_outlook_and_conclusion.tex:25-45:
       "every k stores all n positions again"). ONE position array, sorted by the hash of the LARGEST k, serves every k:
       the bucket of a shorter k-mer is the contiguous slab of the largest-k hashes that start with it, found through the
       same directory. Device memory of the elements falls by about the number of ks; results are identical. The price:
       inside a slab the positions are ordered by the following symbols, not by position, so every result seeded from a
       shorter k is sorted per query after it is written (exact-length and sub-k lookups of short k return whole slabs:
       expect those to be many times slower than with per-k arrays; DESIGN.md section 8 has the numbers). Implies
       KMER_B200_FLAG_NO_AUX. Single device, unsharded. Ignored for one k. */
    KMER_B200_FLAG_SHARED_POSITIONS = 2
};

typedef struct kmer_b200_config {
    int32_t device;        /* CUDA device ordinal; -1 = the calling thread's current device */
    uint32_t mode;         /* default kmer_b200_mode for searches */
    void *stream;          /* cudaStream_t all work is enqueued on; NULL = a private non-blocking stream */
    /* Position-range sharding (multi-GPU). `ranks` passed to create is the slice
       [shard_begin, shard_begin + n) of a text of n_total symbols; the last `halo` symbols of the slice
       belong to the next shard and are only read to complete matches that start in this shard.
       Single-GPU: shard_begin = 0, n_total = 0 (meaning n), halo = 0. */
    uint64_t shard_begin;
    uint64_t n_total;
    uint32_t halo;
    uint32_t directory_bits; /* 0 = automatic; otherwise log2 of the directory size cap per element */
    uint32_t profile;        /* 1 = bracket every kernel launch with CUDA events (kmer_b200_stats);
                                2 = additionally count the 32-byte sectors each search gathers */
    uint32_t reserved;       /* flag bits, KMER_B200_FLAG_* below */
    /* Key-range parts (multi-GPU build of a REPLICATED index). key_parts > 1: `ranks` is the whole text, but every
       element indexes only the k-mers whose hash lies in part key_part of key_parts equal slices of [0, sigma^k):
       1/key_parts of the sorting work per GPU. The parts are concatenated into the full index (part r's position
       array behind part r-1's, directory entries offset by the k-mers of the earlier parts) and handed back with
       kmer_b200_adopt_element; until then the index answers with the hits of its own part only. 32-bit hashes,
       dense directories. 0 or 1: the whole key space. */
    uint32_t key_part;
    uint32_t key_parts;
    /* Several GPUs behind ONE handle, one process (n_devices > 1; `device` is then ignored): kmer_b200_create builds
       a key-range part on each device in parallel (one host thread per device), exchanges the parts between the devices
       over peer copies (NVLink) so that every device holds the whole index, and kmer_b200_search_batch stripes a host
       batch over the devices -- each uploads its slice of the queries over its own PCIe link, searches it, and returns
       its slice of the result. The entry points that take device pointers are not available on such a handle. */
    const int32_t *device_ids;
    uint32_t n_devices;
} kmer_b200_config;

typedef struct kmer_b200_index kmer_b200_index;
typedef struct kmer_b200_result kmer_b200_result;

void kmer_b200_config_default(kmer_b200_config *cfg);
int kmer_b200_abi_version(void);
const char *kmer_b200_last_error(void);

/* ---- build: replaces kmer::kmer_index<alphabet, position_t, ks...>::kmer_index(text, n_threads)
   (kmer_index.hpp:480-496), i.e. kmer_index_element<k>::create for every k (kmer_index.hpp:154-179)
   plus choose_search_scheme (kmer_index.hpp:407-476).
   ranks: n symbol ranks, one byte each, in [0, sigma) -- the memory layout of std::vector<alphabet_t>
   for seqan3 alphabets. ks: the template parameter pack ks... in template order. The caller's buffer is
   not referenced after the call returns. */
int kmer_b200_create(const uint8_t *ranks, uint64_t n, uint32_t sigma, const uint32_t *ks, uint32_t n_ks,
                     const kmer_b200_config *cfg, kmer_b200_index **out);

/* Same, with `d_ranks` already resident in device memory (used to time the build without the H2D copy). */
int kmer_b200_create_from_device(const uint8_t *d_ranks, uint64_t n, uint32_t sigma, const uint32_t *ks,
                                 uint32_t n_ks, const kmer_b200_config *cfg, kmer_b200_index **out);

/* Character input (the step before the path: real texts are characters, e.g. FASTA records). lut256 maps every
   byte value to its rank; bytes that are not in the alphabet must map to a value >= sigma and make the call
   fail with KMER_B200_ERR_INVALID_RANK. The translation runs on the device, fused in front of the packing. */
int kmer_b200_create_from_text(const char *text, uint64_t n, const uint8_t *lut256, uint32_t sigma, const uint32_t *ks,
                               uint32_t n_ks, const kmer_b200_config *cfg, kmer_b200_index **out);
int kmer_b200_search_batch_text(kmer_b200_index *index, const char *q_chars, const uint64_t *q_offsets,
                                uint64_t n_queries, const uint8_t *lut256, uint32_t mode, kmer_b200_result **out);

/* FASTA / FASTQ input (SURVEY.md 8f.3). The file's bytes are parsed on the device: header lines, line breaks (FASTQ: the
   '+' and quality lines too) are dropped, sequence characters are translated through lut256 (a character outside the
   alphabet fails with KMER_B200_ERR_INVALID_RANK), all records are concatenated into one rank text that stays in device
   memory -- feed it to kmer_b200_create_from_device -- and a record table maps positions back. format: 0 = by the
   first byte ('>' / ';' FASTA, '@' FASTQ), 1 = FASTA, 2 = FASTQ (four lines per record; blank lines at the end of the
   file are no records). */
typedef struct kmer_b200_records kmer_b200_records;
int kmer_b200_parse_sequences(const char *data, uint64_t n_bytes, const uint8_t *lut256, uint32_t sigma, uint32_t format,
                              const kmer_b200_config *cfg, kmer_b200_records **out);
uint64_t kmer_b200_records_count(const kmer_b200_records *r);
uint64_t kmer_b200_records_symbols(const kmer_b200_records *r);            /* length of the concatenated text */
const uint64_t *kmer_b200_records_starts(const kmer_b200_records *r);      /* host, [count + 1]: first symbol of each record */
const uint64_t *kmer_b200_records_header_offsets(const kmer_b200_records *r); /* host, [count]: byte offset of the record's header
                                                                              line in `data`; UINT64_MAX for a headerless first record */
const uint8_t *kmer_b200_records_ranks_device(const kmer_b200_records *r); /* device, [symbols] */
/* positions (as returned by a search on the concatenated text) -> record index and offset inside it. query_len > 0:
   a match that runs over the end of its record is not a match of any sequence: record_out = UINT32_MAX for it. */
int kmer_b200_records_locate(const kmer_b200_records *r, const uint32_t *positions, uint64_t n, uint64_t query_len,
                             uint32_t *record_out, uint32_t *offset_out);
void kmer_b200_records_free(kmer_b200_records *r);

/* ---- sequence collections: an index plus a record table starts[0..R] (starts[0] = 0, non-decreasing, starts[R] = n;
   empty records allowed). On a collection index a window [p, p+m) exists only inside one record (no record start s with
   p < s < p + m), so every search returns what searching each record on its own would, positions offset by the
   record's start (seqan3: a search over a collection, reference id = record). An index without records is unchanged.
   - Approximate search (every entry point, strategy and distances) honours the boundaries.
   - Exact search (_search_batch, _ptrs, _text, _batch_device, _count_batch_device) runs in CORRECT mode, as approximate
     search with max_mismatches = 0; mode UINT32_MAX means CORRECT, KMER_B200_MODE_REFERENCE_EXACT is refused with
     KMER_B200_ERR_INVALID_ARGUMENT (the reference has no collections).
   - Host batches take the single-copy staging (kmer_b200_last_search_host_path reports 0): the chunked pipeline does not
     serve collections.
   - The cross-shard and routed entry points (presence_batch_device, search_batch_device_global, search_sharded_*,
     route_*, search_routed_device, unroute_device) return KMER_B200_ERR_UNSUPPORTED.
   - kmer_b200_save writes file version 4 (version 3 plus the table); kmer_b200_load rebuilds it.
   The device holds the table and a bitmap of the record starts (n / 8 bytes), counted by kmer_b200_device_bytes. */
/* Attach the table once: KMER_B200_ERR_INVALID_ARGUMENT for null pointers, n_records = 0 or >= 2^32, starts[0] != 0, a
   decreasing entry, starts[R] != n or records already attached; KMER_B200_ERR_UNSUPPORTED on the handles approximate
   search refuses. kmer_b200_records_starts / _count of a parsed file fit as they are. */
int kmer_b200_attach_records(kmer_b200_index *index, const uint64_t *starts, uint64_t n_records);
/* The host copy of the table ([*n_records + 1]), or NULL (and *n_records = 0) for an index without records. */
const uint64_t *kmer_b200_index_records(const kmer_b200_index *index, uint64_t *n_records);
/* positions -> record (the last r with starts[r] <= p) and offset p - starts[r]; a position >= n gives UINT32_MAX and 0.
   kmer_b200_locate takes host arrays, kmer_b200_locate_device device arrays (a kernel on the index's stream).
   KMER_B200_ERR_INVALID_ARGUMENT on an index without records. */
int kmer_b200_locate(kmer_b200_index *index, const uint32_t *positions, uint64_t n, uint32_t *record_out, uint32_t *offset_out);
int kmer_b200_locate_device(kmer_b200_index *index, const uint32_t *d_positions, uint64_t n, uint32_t *d_record_out,
                            uint32_t *d_offset_out);

void kmer_b200_destroy(kmer_b200_index *index);

/* ---- serialization: construct once, load later (the thesis assumes it, thesis/content/02_implementation.tex:44-46,
   the reference ships no code for it). The file holds the packed text and every element's CSR arrays; load
   restores the index without rebuilding. cfg (device, stream, mode, profile) applies to the loaded index; its
   shard geometry comes from the file. */
int kmer_b200_save(kmer_b200_index *index, const char *path);
int kmer_b200_load(const char *path, const kmer_b200_config *cfg, kmer_b200_index **out);

/* ---- search: replaces kmer_index::search(std::vector<alphabet_t>&) (kmer_index.hpp:505-558) followed
   by kmer_index_result::to_vector() (kmer_index_result.hpp:244-260), for a batch of Q queries.
   q_ranks: all queries' ranks back to back; q_offsets[Q+1]: start of each query in q_ranks.
   The result holds, in host memory, offsets[Q+1], the per-query ascending hit positions back to back,
   and status[Q] (kmer_b200_query_status). mode: a kmer_b200_mode, or UINT32_MAX for the index default.
   Batches of 256 MiB or more are cut into chunks that are uploaded, searched and downloaded concurrently; for 2- and
   4-bit alphabets the library's host threads pack part of the chunks before they cross PCIe (all of them when the
   buffers are pageable), the copy engine moves the rest as they are (DESIGN.md section 7, "Host path"). The buffers may
   be pinned or pageable; they are only read, and only during the call. A collection index (kmer_b200_attach_records)
   answers in CORRECT mode, with hits inside one record only. */
int kmer_b200_search_batch(kmer_b200_index *index, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t n_queries,
                           uint32_t mode, kmer_b200_result **out);

/* Same for queries that live in separate host buffers (std::vector<std::vector<alphabet_t>>): q_ptrs[i] points to the
   q_lens[i] ranks of query i. The library gathers them with its host thread pool -- no per-symbol copy by the caller. */
int kmer_b200_search_batch_ptrs(kmer_b200_index *index, const uint8_t *const *q_ptrs, const uint64_t *q_lens,
                                uint64_t n_queries, uint32_t mode, kmer_b200_result **out);

/* Same with queries resident in device memory and the result left in device memory.
   max_query_len must be >= the longest query in the batch. */
int kmer_b200_search_batch_device(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                  uint64_t n_queries, uint64_t max_query_len, uint32_t mode, kmer_b200_result **out);

/* Count-only variant of the device search (no position list is materialised); the reference analogue is
   timing search() without to_vector(), as its benchmarks do (benchmarks/just_k/main.cpp:58-62). */
int kmer_b200_count_batch_device(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                 uint64_t n_queries, uint64_t max_query_len, uint32_t mode, kmer_b200_result **out);

/* ---- approximate search (no reference analogue): for each query q of length m, every position p, ascending, with
   p + m <= n and at most max_mismatches substituted symbols between T[p, p+m) and q (Hamming distance; no insertions or
   deletions, no window past the end of the text). max_mismatches <= 8, else KMER_B200_ERR_INVALID_ARGUMENT. The search
   seeds from max_mismatches + 1 disjoint exact pieces of the query through the index and verifies every candidate
   window on the packed text (DESIGN.md section 5, "Approximate search"). Per-query status: KMER_B200_QUERY_UNDEFINED for
   an empty query, else OK; a query of m <= max_mismatches symbols matches every window. max_mismatches = 0 gives the
   result of KMER_B200_MODE_CORRECT search. Not available (KMER_B200_ERR_UNSUPPORTED) on a multi-device handle, a
   position-range shard, a shared-positions index or a key-range part that has not been adopted. Query length is
   bounded by the shared-memory staging as for exact search. Same host buffers and result layout as
   kmer_b200_search_batch; the whole batch is staged on the device in one copy. This and the two device forms below
   are the _ex forms (hit strategies, below) with options {max_mismatches, KMER_B200_HITS_ALL, 0, 0}. */
int kmer_b200_search_approx_batch(kmer_b200_index *index, const uint8_t *q_ranks, const uint64_t *q_offsets,
                                  uint64_t n_queries, uint32_t max_mismatches, kmer_b200_result **out);

/* Same with queries resident in device memory and the result left in device memory (max_query_len >= the longest
   query in the batch). */
int kmer_b200_search_approx_batch_device(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                         uint64_t n_queries, uint64_t max_query_len, uint32_t max_mismatches,
                                         kmer_b200_result **out);

/* Count-only variant of the device approximate search (offsets and status; no position list is materialised). */
int kmer_b200_count_approx_batch_device(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                        uint64_t n_queries, uint64_t max_query_len, uint32_t max_mismatches,
                                        kmer_b200_result **out);

/* ---- hit strategies of approximate search (the seqan3 search_cfg::hit_* choices). With d(p) = the Hamming distance
   between T[p, p+m) and the query, H = the hits of kmer_b200_search_approx_batch and d_min = the smallest d(p) over H:
     KMER_B200_HITS_ALL          H
     KMER_B200_HITS_ALL_BEST     the p in H with d(p) = d_min
     KMER_B200_HITS_SINGLE_BEST  the one p in H with the smallest (d(p), p): ties go to the lowest position
     KMER_B200_HITS_STRATA       the p in H with d(p) <= min(e, d_min + strata); strata = 0 is ALL_BEST, >= e is ALL
   Positions are ascending per query; an empty H gives no hits under every strategy. A query of m <= e symbols has
   d_min < m if some window is within m - 1 substitutions, else d_min = m (every window; none when m > n). Statuses as
   for kmer_b200_search_approx_batch. Every strategy other than ALL runs a best pass first (budget min(e, m - 1) per
   query); ALL_BEST and STRATA then search the queries that have hits again, each with budget min(e, d_min + strata).
   The result carries kmer_b200_result_best_distances (u8[Q]: d_min, 0xFF where H is empty or the status is not OK)
   for every strategy other than ALL, and kmer_b200_result_distances (u8[n_positions]: d(p) of each position, in the
   same order) when KMER_B200_APPROX_DISTANCES is set (the count-only form ignores it). KMER_B200_ERR_INVALID_ARGUMENT
   for null options, e > 8, an unknown strategy or unknown flag bits; the handles kmer_b200_search_approx_batch refuses
   are refused the same way. Host batches are staged in one copy; kmer_b200_last_search_transfer counts the two
   arrays. */
typedef enum kmer_b200_approx_hits {
    KMER_B200_HITS_ALL = 0,
    KMER_B200_HITS_ALL_BEST = 1,
    KMER_B200_HITS_SINGLE_BEST = 2,
    KMER_B200_HITS_STRATA = 3
} kmer_b200_approx_hits;

enum { KMER_B200_APPROX_DISTANCES = 1 }; /* kmer_b200_approx_options.flags */

typedef struct kmer_b200_approx_options {
    uint32_t max_mismatches; /* e <= 8 */
    uint32_t hits;           /* kmer_b200_approx_hits */
    uint32_t strata;         /* s, KMER_B200_HITS_STRATA only */
    uint32_t flags;          /* KMER_B200_APPROX_DISTANCES: return d(p) per hit (ignored by the count-only form) */
} kmer_b200_approx_options;

int kmer_b200_search_approx_batch_ex(kmer_b200_index *index, const uint8_t *q_ranks, const uint64_t *q_offsets,
                                     uint64_t n_queries, const kmer_b200_approx_options *options, kmer_b200_result **out);
int kmer_b200_search_approx_batch_device_ex(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                            uint64_t n_queries, uint64_t max_query_len,
                                            const kmer_b200_approx_options *options, kmer_b200_result **out);
int kmer_b200_count_approx_batch_device_ex(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                           uint64_t n_queries, uint64_t max_query_len,
                                           const kmer_b200_approx_options *options, kmer_b200_result **out);

/* ---- k-mer seeding (the reference's kmer_index_element::search_k, kmer_index.hpp:182-190, for every k-mer of every
   query in one call): for each query q of length m and each offset j in [0, m - k], every text position p with
   T[p, p+k) = q[j, j+k). k must be one of the index's ks (auxiliary elements do not count), else
   KMER_B200_ERR_INVALID_ARGUMENT. On a collection index only windows inside one record count. A query shorter than k has
   no k-mers and no hits; every status is KMER_B200_QUERY_OK; a rank >= sigma fails the call with
   KMER_B200_ERR_INVALID_RANK. A query's hits are ordered by (j, p) ascending, and kmer_b200_result_seed_offsets gives
   the j of each one. kmer_b200_result_kmer_counts holds one u32 per k-mer of the batch (sum over q of max(0, m_q - k + 1)
   entries, query order then j order): the k-mer's occurrence count (in-record occurrences on a collection index).
   max_occ > 0 is a repeat cap: a k-mer with more than max_occ occurrences contributes no hits, and its count entry reads
   max_occ + 1. max_occ = 0: no cap. Query length is not bounded by a shared-memory staging (each query is walked in
   tiles); j is reported in 32 bits, so max_query_len < 2^32. Refused (KMER_B200_ERR_UNSUPPORTED) on the handles
   approximate search refuses. The host form stages the batch in one copy (counted by kmer_b200_last_search_transfer);
   the device forms take max_query_len >= the longest query; the count-only form returns offsets, status and the k-mer
   counts but no positions. */
int kmer_b200_seed_batch(kmer_b200_index *index, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t n_queries,
                         uint32_t k, uint32_t max_occ, kmer_b200_result **out);
int kmer_b200_seed_batch_device(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                uint64_t n_queries, uint64_t max_query_len, uint32_t k, uint32_t max_occ,
                                kmer_b200_result **out);
int kmer_b200_count_seeds_batch_device(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                       uint64_t n_queries, uint64_t max_query_len, uint32_t k, uint32_t max_occ,
                                       kmer_b200_result **out);

/* ---- record votes: which records of a collection index each read comes from (the question behind k-mer classifiers,
   strain or transcript assignment and contamination screening). For read q of length m and each j in [0, m - k], occ(j)
   is the number of in-record occurrences of q[j, j+k) (exactly seeding's uncapped k-mer count). k-mer j is counted when
   occ(j) >= 1 and, with max_occ > 0, occ(j) <= max_occ. recs(j) is the set of records its occurrences lie in (the record
   of position p is the last r with starts[r] <= p, the rule of kmer_b200_locate, so empty records get no votes), and
   votes(q, r) = #{counted j : r in recs(j)}: a k-mer occurring five times in one record gives it one vote, the same
   k-mer at two offsets of the read gives two. Per read, every (record, votes) with votes >= min_votes, ordered by votes
   descending, then record ascending: kmer_b200_result_positions holds the RECORD IDS of this result, and
   kmer_b200_result_votes their votes ([n_positions]); kmer_b200_result_kmer_hits gives each read's number of counted
   k-mers ([n_queries]). Exact for any number of records a read hits (reads beyond a shared-memory table take a
   global-memory path); running out of device memory is KMER_B200_ERR_OUT_OF_MEMORY, never a truncated list.
   Every status is KMER_B200_QUERY_OK; a read shorter than k has no entries and 0 k-mer hits; a rank >= sigma anywhere
   fails the call with KMER_B200_ERR_INVALID_RANK. KMER_B200_ERR_INVALID_ARGUMENT: an index without records, k not one
   of the index's ks (auxiliary elements do not count), min_votes = 0, null pointers. KMER_B200_ERR_UNSUPPORTED on the
   handles seeding refuses (multi-device handles, position-range shards, key-range parts not yet adopted). The host form
   stages the batch in one copy; the device form takes max_query_len >= the longest read (reads are walked in tiles, so
   their length is not otherwise bounded). Reverse complements are not considered: pass one as a read of its own. */
int kmer_b200_record_votes(kmer_b200_index *index, const uint8_t *q_ranks, const uint64_t *q_offsets, uint64_t n_queries,
                           uint32_t k, uint32_t max_occ, uint32_t min_votes, kmer_b200_result **out);
int kmer_b200_record_votes_device(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                  uint64_t n_queries, uint64_t max_query_len, uint32_t k, uint32_t max_occ, uint32_t min_votes,
                                  kmer_b200_result **out);

/* ---- k-mer spectrum: what the index holds as a whole, read off the bucket sizes of the element of k (one of the index's
   ks, views of a shared-positions index included; auxiliary elements do not count, any other k is
   KMER_B200_ERR_INVALID_ARGUMENT). The counted windows are p in [0, n - k]; on a collection index only those inside one
   record. count(h) is the number of counted windows with hash h: the uncapped count seeding reports for that k-mer.
   Refused (KMER_B200_ERR_UNSUPPORTED) on multi-device handles, position-range shards and key-range parts that have not
   been adopted. Runs on the index's stream and returns when the results are on the host. */
typedef struct kmer_b200_spectrum_info {
    uint64_t total;      /* counted windows */
    uint64_t distinct;   /* #{h : count(h) >= 1} */
    uint64_t max_count;  /* the largest count(h), 0 when nothing is counted */
    uint64_t key_space;  /* sigma^k, saturated at UINT64_MAX */
} kmer_b200_spectrum_info;
/* hist[c] = #{h : count(h) = c} for 1 <= c < n_bins - 1, hist[n_bins - 1] = #{h : count(h) >= n_bins - 1},
   hist[0] = sigma^k - distinct (saturated). n_bins >= 2; hist may be NULL (info only), info may be NULL. */
int kmer_b200_spectrum(kmer_b200_index *index, uint32_t k, uint64_t *hist, uint64_t n_bins, kmer_b200_spectrum_info *info);
/* Every h with count(h) >= min_count (>= 1), ordered by count descending, then hash ascending: *n_out = how many exist
   (N), and the first min(N, cap) go to hashes / counts (host arrays; NULL allowed when cap = 0). Jellyfish-style "top
   100" is min_count = 1, cap = 100. */
int kmer_b200_frequent_kmers(kmer_b200_index *index, uint32_t k, uint64_t min_count, uint64_t *hashes, uint64_t *counts,
                             uint64_t cap, uint64_t *n_out);
/* The repeat cutoff that ignores the most frequent fraction of the distinct k-mers: the smallest c >= 1 with
   #{h : count(h) > c} <= floor(fraction * distinct), 0 when distinct = 0. fraction in [0, 1). Exact at any count;
   seeding with max_occ = cutoff drops exactly the k-mers above it. */
int kmer_b200_occurrence_cutoff(kmer_b200_index *index, uint32_t k, double fraction, uint64_t *cutoff);

uint64_t kmer_b200_result_n_queries(const kmer_b200_result *r);
uint64_t kmer_b200_result_n_positions(const kmer_b200_result *r);
int kmer_b200_result_on_device(const kmer_b200_result *r);
/* Device-resident results only (else NULL): a device array u32[1 + n_queries]; element 0 = number n of queries the
 * count pass found hits for, elements 1..n = their ids in no particular order. A listed query can still have an
 * empty result (sharded search: the whole-text presence rule is applied after the count pass). Lets a caller that
 * merges per-shard results touch only the queries that have something to merge. */
const uint32_t *kmer_b200_result_hit_queries(const kmer_b200_result *r);
const uint64_t *kmer_b200_result_offsets(const kmer_b200_result *r);   /* [Q+1] */
const uint32_t *kmer_b200_result_positions(const kmer_b200_result *r); /* [offsets[Q]], NULL if count-only */
const uint8_t *kmer_b200_result_status(const kmer_b200_result *r);     /* [Q] */
const uint8_t *kmer_b200_result_distances(const kmer_b200_result *r);      /* [n_positions] or NULL (approximate search) */
const uint8_t *kmer_b200_result_best_distances(const kmer_b200_result *r); /* [Q] or NULL (approximate search) */
const uint32_t *kmer_b200_result_seed_offsets(const kmer_b200_result *r);  /* [n_positions] or NULL (seeding, not count-only) */
const uint32_t *kmer_b200_result_kmer_counts(const kmer_b200_result *r);   /* [n_kmers] or NULL (seeding) */
uint64_t kmer_b200_result_n_kmers(const kmer_b200_result *r);              /* k-mers of a seeding batch, else 0 */
const uint32_t *kmer_b200_result_votes(const kmer_b200_result *r);         /* [n_positions] or NULL (record votes) */
const uint32_t *kmer_b200_result_kmer_hits(const kmer_b200_result *r);     /* [n_queries] or NULL (record votes) */
void kmer_b200_result_free(kmer_b200_result *r);

/* ---- sharded (multi-GPU) search, two phases around one cross-rank exchange.
   Phase A fills d_present[Q] with one flag per indexed part of the query (part j occurs in this shard); the
   caller combines the flags of all shards over NCCL and passes the result to phase B
   (kmer_b200_search_batch_device_global), which then reproduces the reference's whole-text early-return /
   throw decisions (kmer_index.hpp:216-227, :119-122) on every shard.
   present_format 0: uint64_t per query, bit j = part j (combine with bitwise OR; up to 64 parts);
   present_format 1: uint32_t per query, bit 4j = part j (combine with a SUM all-reduce over <= 15 shards --
                     NCCL has no bitwise OR; up to 8 parts per query, longer queries report no hits). */
int kmer_b200_presence_batch_device(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                    uint64_t n_queries, uint64_t max_query_len, uint32_t mode, void *d_present,
                                    uint32_t present_format);
int kmer_b200_search_batch_device_global(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                         uint64_t n_queries, uint64_t max_query_len, uint32_t mode,
                                         const void *d_present_global, uint32_t present_format, kmer_b200_result **out);

/* Fused form of the two phases (presence flags in format 1 only): begin runs the count pass and writes this
   shard's flags to d_present4[Q]; the caller SUM-all-reduces them; finish applies the whole-text rule, then
   scans and writes the positions. One pass over the queries less than presence + search_global. */
typedef struct kmer_b200_pending kmer_b200_pending;
int kmer_b200_search_sharded_begin(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets,
                                   uint64_t n_queries, uint64_t max_query_len, uint32_t mode, uint32_t *d_present4,
                                   kmer_b200_pending **out);
int kmer_b200_search_sharded_finish(kmer_b200_pending *pending, const uint32_t *d_present4_global, kmer_b200_result **out);
/* Gives up a search begun with kmer_b200_search_sharded_begin (e.g. the cross-rank exchange failed): releases its
   device buffers. finish consumes the handle too; call exactly one of the two. */
void kmer_b200_search_sharded_abort(kmer_b200_pending *pending);
/* Between begin and finish: this shard's per-query hit counts with the whole-text rule applied (u64[Q], valid until
   finish turns them into offsets) and the list of queries the count pass found hits for (as
   kmer_b200_result_hit_queries). Lets a shard send its sparse (query id, count) pairs to the merging shard before
   its own scan and write pass run. Both are device pointers owned by the pending search. */
int kmer_b200_search_sharded_peek(kmer_b200_pending *pending, const uint32_t *d_present4_global,
                                  const uint64_t **d_counts_out, const uint32_t **d_hit_queries_out);
/* Merging on the shard that assembles the result (optional, between begin and finish): add another shard's
   per-query hit counts -- n (query id, count) pairs, device arrays -- to this shard's counts. d_within_out[i]
   receives what the count of query d_ids[i] was before the call: with calls made in rank order, the offset of that
   shard's list inside the query's merged list. After finish, the result's offsets are the merged offsets,
   n_positions the merged total, this shard's own hits are already in place at the head of every query's range, and
   the caller copies the other shards' lists to offsets[id] + within. */
int kmer_b200_search_sharded_add_counts(kmer_b200_pending *pending, const uint32_t *d_present4_global,
                                        const int64_t *d_ids, const int64_t *d_counts, uint64_t n, int64_t *d_within_out);

/* ---- key-range parts: export a part, adopt the assembled whole (see kmer_b200_config.key_parts) */
typedef struct kmer_b200_part {
    uint64_t key_lo, key_hi;     /* the hashes this part indexes: [key_lo, key_hi) */
    uint64_t n_kmers;            /* k-mers in the part = length of d_positions */
    uint64_t directory_entries;  /* key_hi - key_lo + 1 (dense); entry j = number of the part's k-mers with hash - key_lo < j */
    const uint32_t *d_positions; /* device, stably sorted by hash */
    const uint32_t *d_directory; /* device */
} kmer_b200_part;
int kmer_b200_element_part(const kmer_b200_index *index, uint32_t element, kmer_b200_part *out);
/* d_dst[j] = directory[j] + base for j < n (n <= directory_entries): the part's directory as a slice of the whole
   index's, `base` = number of k-mers in the parts before this one. Enqueued on the index's stream. */
int kmer_b200_export_directory(kmer_b200_index *index, uint32_t element, uint64_t base, uint64_t n, uint32_t *d_dst);
/* The part's directory as bucket sizes, one byte per hash of [key_lo, key_hi) -- a quarter of the bytes to move between
   GPUs. *n_large_out = buckets holding 255 or more k-mers (their size does not fit: ship the directory itself then). */
int kmer_b200_export_bucket_sizes(kmer_b200_index *index, uint32_t element, uint8_t *d_sizes, uint64_t *n_large_out);
/* The whole directory d_directory[n_keys + 1] from the bucket sizes of all n_keys hashes (exclusive prefix sum; the last
   entry is the total). Runs on the index's stream. */
int kmer_b200_directory_from_sizes(kmer_b200_index *index, const uint8_t *d_sizes, uint64_t n_keys, uint32_t *d_directory);
/* Replace the element's arrays by the assembled whole: d_positions[n_kmers] (n_kmers = n - k + 1) and the dense
   directory d_directory[sigma^k + 1], both device arrays that stay owned by the caller and must outlive the index.
   The element then covers the whole key space. */
int kmer_b200_adopt_element(kmer_b200_index *index, uint32_t element, const uint32_t *d_positions, uint64_t n_kmers,
                            const uint32_t *d_directory, uint64_t directory_entries);
/* Same, with the position array left in the parts the GPUs built ("peer positions"): part r holds the entries
   [part_first[r], part_first[r + 1]) of the whole position array (part_first has n_parts + 1 entries, n_parts <= 8; part
   boundaries are the key-range boundaries, so a bucket never straddles two parts). A part may be another GPU's memory
   mapped into this process (CUDA IPC); the search then reads those candidates over NVLink. Only the directory -- whole,
   d_directory as above -- is replicated: the build moves a byte per bucket between the GPUs instead of the positions.
   The arrays stay the caller's and must outlive the index. */
int kmer_b200_adopt_element_parts(kmer_b200_index *index, uint32_t element, const uint32_t *const *d_position_parts,
                                  const uint64_t *part_first, uint32_t n_parts, const uint32_t *d_directory,
                                  uint64_t directory_entries);
/* Device buffers that other processes (one per GPU) can map: create = a plain device allocation on `device` plus its
   64-byte CUDA IPC handle; open = map a buffer created by another process into this one, readable by kernels running on
   `device` (peer access over NVLink is enabled on the way); release = unmap (opened != 0) or free (opened == 0). These
   carry the position parts of kmer_b200_adopt_element_parts between the ranks of a multi-process job. */
int kmer_b200_peer_buffer_create(int device, uint64_t bytes, void **d_ptr, uint8_t *handle64);
int kmer_b200_peer_buffer_open(int device, const uint8_t *handle64, void **d_ptr);
int kmer_b200_peer_buffer_release(int device, void *d_ptr, int opened);

/* ---- key-range multi-GPU search: the index stays partitioned (one key-range part per GPU, no assembly), queries
   travel to the GPU that owns the hash of their first k symbols and results travel back. Single-k indices with 32-bit
   hashes; queries no shorter than k. Each rank drives these calls and moves the blocks between them with three
   equal-/variable-split all-to-all collectives (kmer_index_b200/sharded.py: search_routed):

     origin   kmer_b200_route_queries_device   its slice of the batch -> n_parts send blocks          --all-to-all-->
     owner    kmer_b200_search_routed_device   received blocks -> search -> return blocks + positions  --all-to-all x2-->
     origin   kmer_b200_unroute_device         return blocks + positions -> CSR result of its slice

   Whole-text rules of the reference (a part of the query absent anywhere => empty; rest too short => throw) are
   decided by the owner from a presence bitmap over the whole key space: every part exports its slice
   (kmer_b200_presence_export), the slices are all-gathered, the whole bitmap is attached (kmer_b200_presence_attach). */
typedef struct kmer_b200_route_plan {
    uint32_t n_parts;            /* GPUs = index parts */
    uint32_t stride;             /* 64-bit words per packed query */
    uint32_t capacity;           /* records per block (the same on every rank) */
    uint32_t reserved;
    uint64_t block_bytes;        /* one send block; send / receive buffers hold n_parts of them */
    uint64_t return_block_bytes; /* one return block */
} kmer_b200_route_plan;
/* n_queries: the largest per-rank batch slice; capacity = n_queries / n_parts * slack + 1024 (slack <= 0: 1.25) */
int kmer_b200_route_plan_make(const kmer_b200_index *index, uint64_t n_queries, uint64_t max_query_len, uint32_t n_parts,
                              double slack, kmer_b200_route_plan *out);
/* d_status[Q]: 0xFF for routed queries, else the status decided at the origin (empty / over-long queries).
   sent_counts[n_parts] (host): records per block; a count above plan->capacity means that block overflowed (nothing
   was lost on the device side only if the caller re-plans with a larger capacity and routes again). */
int kmer_b200_route_queries_device(kmer_b200_index *index, const uint8_t *d_q_ranks, const uint64_t *d_q_offsets, uint64_t n_queries,
                                   uint32_t mode, const kmer_b200_route_plan *plan, uint8_t *d_send_blocks, uint8_t *d_status,
                                   uint32_t *sent_counts);
/* position_splits[n_parts] (host): how many positions of the result belong to each origin, in block order; the result's
   position array is the send buffer of the positions all-to-all. */
int kmer_b200_search_routed_device(kmer_b200_index *index, uint8_t *d_received_blocks, const kmer_b200_route_plan *plan, uint32_t mode,
                                   uint8_t *d_return_blocks, uint64_t *position_splits, kmer_b200_result **out);
int kmer_b200_unroute_device(kmer_b200_index *index, uint8_t *d_send_blocks, uint8_t *d_received_return_blocks,
                             const kmer_b200_route_plan *plan, const uint32_t *sent_counts, const uint32_t *d_received_positions,
                             const uint64_t *received_position_splits, uint64_t n_queries, const uint8_t *d_status,
                             kmer_b200_result **out);
/* bit h of the bitmap = hash h occurs in the text; the bitmap has sigma^k bits rounded up to 64-bit words (+1 word) */
uint64_t kmer_b200_presence_words(const kmer_b200_index *index, uint32_t element);
int kmer_b200_presence_export(kmer_b200_index *index, uint32_t element, uint64_t *d_bitmap);
int kmer_b200_presence_attach(kmer_b200_index *index, uint32_t element, const uint64_t *d_bitmap);

/* ---- introspection (parity tests and roofline accounting) */
typedef struct kmer_b200_element_info {
    uint32_t k;
    uint32_t key_bits;        /* ceil(log2(sigma^k)) */
    uint32_t directory_shift; /* bucket directory is indexed by hash >> shift */
    uint32_t sort_passes;
    uint64_t n_kmers;         /* n - k + 1 */
    uint64_t directory_entries;
    uint64_t device_bytes;
} kmer_b200_element_info;

uint32_t kmer_b200_n_elements(const kmer_b200_index *index);
int kmer_b200_element_info_get(const kmer_b200_index *index, uint32_t element, kmer_b200_element_info *out);
/* Copy element's position array (all k-mer start positions stably sorted by hash: the concatenation of
   the reference's _data buckets in ascending hash order, kmer_index.hpp:52,165) to host memory. */
int kmer_b200_element_positions(kmer_b200_index *index, uint32_t element, uint32_t *out, uint64_t cap);
/* Copy the sorted hash array (one per position above) to host memory. */
int kmer_b200_element_hashes(kmer_b200_index *index, uint32_t element, uint64_t *out, uint64_t cap);
/* Row m of the scheme table (_optimal_nk_sum[m], _use_multi_search_scheme[m]; kmer_index.hpp:404-476).
   Returns the number of summands and writes up to cap of them. */
uint64_t kmer_b200_scheme(const kmer_b200_index *index, uint64_t m, uint32_t *out_ks, uint64_t cap, int *use_multi);

/* The plan the search runs for a query of length m (SURVEY.md 8f.4): which element seeds the candidate list, how many
   directory lookups it needs, and -- from the bucket statistics measured on THIS index -- how many candidates and
   32-byte sectors that costs for a query whose seed k-mer occurs. mode REFERENCE_EXACT follows the reference's table
   (choose_search_scheme, kmer_index.hpp:407-476) where the result depends on it and otherwise seeds from the largest
   k <= m like CORRECT does; CORRECT always seeds from the largest k <= m (the shortest buckets) and verifies the rest of
   the query against the text, which makes every length as cheap as the exact-k lookup plus one text window. */
typedef struct kmer_b200_plan_row {
    uint32_t m;
    uint32_t kind;      /* 0 exact bucket, 1 prefix slab (m < every usable k), 2 contiguous verify, 3 the reference's plan for
                           >= 3 parts + rest (kmer_index.hpp:314), 4 the reference's multi-k sum plan (:526,535), 5 throws */
    uint32_t seed_k;    /* k of the element that supplies the candidates */
    uint32_t n_lookups; /* directory lookups per query */
    double expected_candidates; /* per query whose seed occurs: mean occupied bucket (or slab) length of the seed element */
    double expected_sectors;    /* lookups + candidate list + text windows, in 32-byte sectors */
} kmer_b200_plan_row;
/* rows for m = m_lo .. m_hi (out has m_hi - m_lo + 1 entries). The first call measures the bucket statistics on the device. */
int kmer_b200_plan_table(kmer_b200_index *index, uint32_t mode, uint32_t m_lo, uint32_t m_hi, kmer_b200_plan_row *out);

/* The same row computed on the host from the ks alone (no device, no index needed). */
uint64_t kmer_b200_scheme_for_ks(const uint32_t *ks, uint32_t n_ks, uint64_t m, uint32_t *out_ks, uint64_t cap,
                                 int *use_multi);

/* Per-kernel accounting since the last reset: launches, device time (CUDA events on the launching
   stream; only when cfg.profile = 1) and the algorithmic bytes the kernel must move (DESIGN.md). */
typedef struct kmer_b200_kernel_stat {
    const char *name;
    uint64_t launches;
    double device_ms;
    double algorithmic_bytes;
} kmer_b200_kernel_stat;

uint32_t kmer_b200_stats(kmer_b200_index *index, kmer_b200_kernel_stat *out, uint32_t cap);
void kmer_b200_stats_reset(kmer_b200_index *index);
uint64_t kmer_b200_device_bytes(const kmer_b200_index *index);

/* profile = 2 only: number of 32-byte sectors at data-dependent addresses (directory slots, bucket entries,
   text windows) the last search had to gather -- the algorithmic work of the search kernel. */
/* Debug aid (no reference analogue). With KMER_B200_GUARD=1 in the environment every device allocation of the library
   is bracketed by two 4 KB canary zones that are verified on the device when the allocation is freed: the number of
   damaged canary bytes seen so far, i.e. stores that landed just outside a buffer. 0 without the variable. The selftest
   makes two such stores on purpose and checks that they are counted. */
uint64_t kmer_b200_debug_guard_violations(void);
int kmer_b200_debug_guard_selftest(void);
uint64_t kmer_b200_last_search_gathers(const kmer_b200_index *index);
/* Bytes the last kmer_b200_search_batch / _ptrs / _text on this handle moved over PCIe: host to device (ranks as they are
   or packed, offsets or 16-bit lengths -- whichever the call chose) and device to host (offsets, status, positions). */
void kmer_b200_last_search_transfer(const kmer_b200_index *index, uint64_t *h2d_bytes, uint64_t *d2h_bytes);
/* Bytes the text took over PCIe when the index was built from a host buffer (large 2- / 4-bit texts are partly packed on
   the host threads first); 0 for an index built from device memory or loaded from a file. */
uint64_t kmer_b200_build_transfer(const kmer_b200_index *index);
/* Which host pipeline that call took: 0 = one copy each way (small batches), 3 = chunks, packed as a stream on the host
   threads, raw_pct percent of them sent as 1-byte ranks at the same time (100: every chunk raw; pack_gbs = the host's
   measured streaming pack rate, 0 when not needed). The codes 1 and 2 are no longer reported. */
void kmer_b200_last_search_host_path(const kmer_b200_index *index, uint32_t *pipeline, uint32_t *raw_pct, double *pack_gbs);
/* Calibration of the random-gather ceiling: n_gathers independent 8-byte reads at random addresses of a
   table_bytes table (>> L2); *ms_out = device time. sectors/s = n_gathers / time. */
int kmer_b200_gather_probe(uint64_t table_bytes, uint64_t n_gathers, void *stream, double *ms_out);
/* The same probe over a table the caller provides (device memory of this GPU, or another GPU's memory mapped with
   kmer_b200_peer_buffer_open: the random-read rate over NVLink). */
int kmer_b200_gather_probe_at(const void *d_table, uint64_t table_bytes, uint64_t n_gathers, void *stream, double *ms_out);

/* Host-side helper of kmer_b200_search_batch, exposed for tests and for callers that keep batches packed: n ranks
   (1 byte each) -> the device's b-bit MSB-first words (b = 2 for sigma <= 4, 4 for sigma <= 16, else 8), query
   boundaries ignored; packed with all threads of the library's host pool. words must hold
   kmer_b200_host_pack_stream_words(n, sigma) entries. Returns KMER_B200_ERR_INVALID_RANK when a rank >= sigma was seen.
   Needs no device. */
uint64_t kmer_b200_host_pack_stream_words(uint64_t n, uint32_t sigma);
int kmer_b200_host_pack_stream(const uint8_t *ranks, uint64_t n, uint32_t sigma, uint64_t *words);

/* ---- scalar helpers kept from the reference API */
/* kmer::detail::fast_pow (fast_pow.hpp:46-93): base^exp mod 2^64, 0 when exp >= 63 and base != 1 */
uint64_t kmer_b200_fast_pow(uint64_t base, uint8_t exp);
/* the k-mer hash sum_i rank_i * sigma^(k-1-i) (kmer_index.hpp:56-73) */
uint64_t kmer_b200_hash(const uint8_t *ranks, uint32_t k, uint32_t sigma);
/* choose_best_k (choose_best_k.hpp:12-60); ties keep the candidate order (stable) */
uint64_t kmer_b200_choose_best_k(const uint64_t *query_lengths, uint64_t n_lengths, uint64_t n_k, uint64_t *out_ks);

/* ---- synthetic inputs on the device (bench.py; SURVEY.md 8d): counter-based SplitMix64, identical to
   kmer_index_b200/synth.py */
int kmer_b200_synth_ranks_device(uint8_t *d_out, uint64_t n, uint64_t start, uint32_t sigma, uint64_t seed, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* KMER_B200_H */
