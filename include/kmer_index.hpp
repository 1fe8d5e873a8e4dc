// kmer_index.hpp -- header-only C++ API of the B200 k-mer index.
//
// Source-compatible with the reference's public surface (Clemapfel/kmer_index, kmer_index.hpp):
//
//   kmer::kmer_index<alphabet_t, position_t, ks...>(text, n_threads)      kmer_index.hpp:350-352, 480-496
//   kmer::make_kmer_index<ks...>(text, n_threads)                         kmer_index.hpp:569-579
//   index.search(query) -> kmer::detail::kmer_index_result<position_t>    kmer_index.hpp:505-558
//   result.to_vector()                                                    kmer_index_result.hpp:244-260
//   kmer::detail::fast_pow(base, exp)                                     fast_pow.hpp:46-93
//
// plus kmer::single_kmer_index<k> / kmer::multi_kmer_index<ks...> (the thesis' names) and the batched entry
// point search_batch(), which is what a GPU wants to be fed. Everything heavy happens in libkmer_b200.so
// (include/kmer_b200.h); this header only converts alphabets to ranks and results to vectors.
// Link with -lkmer_b200. There is no CPU fallback: construction throws std::runtime_error without a device.
//
// Differences from the reference, all deliberate:
//   * the result OWNS its sorted positions (the reference's holds pointers into the index);
//     size() is the number of hits (the reference's returns 0 for bypass results, a defect);
//     begin()/end() iterate the positions (the reference's iterator does not compile).
//   * search(std::vector<alphabet_t>&&) returns its result (the reference's has no return statement).
//   * n_threads is accepted and ignored; extend_query_size_range() is rejected above 10000.
//   * texts and queries held in contiguous storage of 1-byte alphabet objects (std::vector<kmer::dna4>, seqan3
//     alphabets) are handed to the library as they are -- the object's byte IS its rank -- without a per-symbol copy.
//   * search_batch() returns views of the library's result buffers (kmer_batch_result keeps them alive; .to_vector() on
//     a view copies it) and collects the queries' pointers on all host cores: 10^8 queries in a
//     std::vector<std::vector<dna4>> take 0.47 s, 63 ms of it inside the library (profiles/r02/header_bench.txt).
//   * an index can span several GPUs: kmer_index(text, devices) builds it from key-range parts on all of them and
//     search_batch() stripes the batch over them (kmer_b200_config.device_ids).
//   * kmer_index(texts, kmer::collection) indexes a collection of texts: no hit spans two of them, locate() gives (text, offset).
//   * the alphabet requirement is `a.to_rank()` plus kmer::alphabet_size<A>; seqan3 alphabets satisfy it when
//     seqan3 is available, kmer::dna4 / dna5 / dna15 / aa27 below are rank-only stand-ins.
#pragma once

#include <algorithm>
#include <array>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <memory>
#include <ranges>
#include <stdexcept>
#include <string>
#include <thread>
#include <type_traits>
#include <utility>
#include <vector>

#include "kmer_b200.h"

#if __has_include(<seqan3/alphabet/concept.hpp>)
#include <seqan3/alphabet/concept.hpp>
#define KMER_B200_HAVE_SEQAN3 1
#endif

namespace kmer
{
    // ------------------------------------------------------------------------------------------ alphabets
    template<std::size_t SIGMA>
    struct rank_alphabet
    {
        static constexpr std::size_t alphabet_size = SIGMA;
        std::uint8_t rank{0};
        constexpr std::uint8_t to_rank() const noexcept { return rank; }
        constexpr rank_alphabet& assign_rank(std::uint8_t r) noexcept { rank = r; return *this; }
        friend constexpr bool operator==(rank_alphabet a, rank_alphabet b) noexcept { return a.rank == b.rank; }
        friend constexpr bool operator!=(rank_alphabet a, rank_alphabet b) noexcept { return a.rank != b.rank; }
    };
    using dna4 = rank_alphabet<4>;
    using dna5 = rank_alphabet<5>;
    using dna15 = rank_alphabet<15>;
    using aa27 = rank_alphabet<27>;

    namespace detail
    {
        template<typename T, typename = void>
        struct alphabet_size_of;
        template<typename T>
        struct alphabet_size_of<T, std::void_t<decltype(T::alphabet_size)>>
        { static constexpr std::size_t value = T::alphabet_size; };
#ifdef KMER_B200_HAVE_SEQAN3
        template<typename T>
            requires (!requires { T::alphabet_size; }) && seqan3::alphabet<T>
        struct alphabet_size_of<T, void>
        { static constexpr std::size_t value = seqan3::alphabet_size<T>; };
#endif
    }

    template<typename T>
    inline constexpr std::size_t alphabet_size = detail::alphabet_size_of<std::remove_cvref_t<T>>::value;

    template<typename T>
    concept alphabet = requires(T const a) {
        { a.to_rank() } -> std::convertible_to<std::size_t>;
        { alphabet_size<T> } -> std::convertible_to<std::size_t>;
    };

    namespace detail
    {
        // fast_pow.hpp:46-93: square-and-multiply mod 2^64; 0 once exp needs more than 6 bits... i.e. exp >= 63
        // (the reference's table returns the "overflow" marker there), except base == 1
        constexpr std::size_t fast_pow(std::size_t base, std::uint8_t exp)
        {
            if (exp >= 63)
                return base == 1 ? 1 : 0;
            std::size_t result = 1;
            while (exp)
            {
                if (exp & 1) result *= base;
                exp >>= 1;
                base *= base;
            }
            return result;
        }

        enum class BYPASS_BITMASK : bool { YES = true, NO = false };   // kmer_index_result.hpp:11 (kept for source compat)

        // kmer_index_result.hpp:14-272. The reference's result points into the index (bucket pointers + a bitmask of
        // usable entries, or the BYPASS flag); this one owns its candidates, keeps the same mask surface
        // (should_use / should_not_use, kmer_index_result.hpp:262-270) and to_vector() filters and sorts as :244-260.
        // Results returned by search() arrive finished: ascending positions, bypass set.
        template<typename position_t>
        class kmer_index_result
        {
            std::vector<position_t> _positions;
            std::vector<bool> _bitmask;           // unused when _bypass
            bool _bypass = true;

        public:
            kmer_index_result() = default;                                                          // :203-205
            explicit kmer_index_result(std::vector<position_t> sorted_positions) : _positions(std::move(sorted_positions)) {}
            // :207-217  one bucket, every entry usable (zero_or_one = true) or not, optionally bypassing the mask
            kmer_index_result(std::vector<position_t> const* bucket, bool zero_or_one = true, BYPASS_BITMASK bypass = BYPASS_BITMASK::NO)
                : _positions(bucket ? *bucket : std::vector<position_t>{}), _bitmask(_positions.size(), zero_or_one),
                  _bypass(bypass == BYPASS_BITMASK::YES) {}
            // :219-236  several buckets, concatenated
            kmer_index_result(std::vector<std::vector<position_t> const*> const& buckets, BYPASS_BITMASK bypass = BYPASS_BITMASK::YES)
                : _bypass(bypass == BYPASS_BITMASK::YES)
            {
                for (auto const* b : buckets)
                    if (b) _positions.insert(_positions.end(), b->begin(), b->end());
                _bitmask.assign(_positions.size(), true);
            }

            void should_use(std::size_t i) { _bitmask.at(i) = true; }                                // :262-265
            void should_not_use(std::size_t i) { _bitmask.at(i) = false; }                           // :267-270

            // number of hits (the reference counts mask bits and so reports 0 for bypass results, a defect: :239-242)
            std::size_t size() const noexcept
            {
                return _bypass ? _positions.size() : std::size_t(std::count(_bitmask.begin(), _bitmask.end(), true));
            }
            bool empty() const noexcept { return size() == 0; }
            std::vector<position_t> to_vector() const                                                // :244-260
            {
                std::vector<position_t> out;
                out.reserve(_positions.size());
                for (std::size_t i = 0; i < _positions.size(); ++i)
                    if (_bypass || _bitmask[i]) out.push_back(_positions[i]);
                if (!std::is_sorted(out.begin(), out.end())) std::sort(out.begin(), out.end());
                return out;
            }
            // iteration over the hits (the reference's iterator does not compile: :98-101,166,182)
            auto begin() const noexcept { return _positions.begin(); }
            auto end() const noexcept { return _positions.end(); }
        };

        // read-only view of an array that a batch result keeps alive (search_batch() hands the library's pinned result
        // buffers out as they are: a batch of 10^8 queries is 0.9 GB that nobody should copy on one thread)
        template<typename T>
        class array_view
        {
            T const* _data = nullptr;
            std::size_t _size = 0;

        public:
            using value_type = T;
            array_view() = default;
            array_view(T const* data, std::size_t size) : _data(data), _size(size) {}
            std::size_t size() const noexcept { return _size; }
            bool empty() const noexcept { return _size == 0; }
            T const* data() const noexcept { return _data; }
            T const* begin() const noexcept { return _data; }
            T const* end() const noexcept { return _data + _size; }
            T const& operator[](std::size_t i) const { return _data[i]; }
            T const& front() const { return _data[0]; }
            T const& back() const { return _data[_size - 1]; }
            std::vector<T> to_vector() const { return std::vector<T>(begin(), end()); }
            friend bool operator==(array_view const& a, array_view const& b)
            {
                return a._size == b._size && std::equal(a.begin(), a.end(), b.begin());
            }
            friend bool operator==(array_view const& a, std::vector<T> const& b)
            {
                return a._size == b.size() && std::equal(a.begin(), a.end(), b.begin());
            }
        };

        // fn(lo, hi) over [0, n) on the host's cores (large batches only: a thread costs more than 10^4 iterations)
        template<typename fn_t>
        void parallel_ranges(std::size_t n, fn_t&& fn)
        {
            std::size_t const n_threads = n < (std::size_t(1) << 18) ? 1 : std::min<std::size_t>(std::max(1u, std::thread::hardware_concurrency()), 32);
            if (n_threads == 1)
                return fn(std::size_t(0), n);
            std::vector<std::thread> workers;
            for (std::size_t t = 0; t < n_threads; ++t)
                workers.emplace_back([&fn, n, t, n_threads] { fn(n * t / n_threads, n * (t + 1) / n_threads); });
            for (auto& w : workers)
                w.join();
        }

        inline void check(int status)
        {
            if (status == KMER_B200_OK)
                return;
            std::string msg = kmer_b200_last_error();
            if (status == KMER_B200_ERR_INVALID_ARGUMENT || status == KMER_B200_ERR_INVALID_RANK)
                throw std::invalid_argument("kmer_b200: " + msg);
            throw std::runtime_error("kmer_b200 (" + std::to_string(status) + "): " + msg);
        }

        // contiguous storage of 1-byte alphabet objects whose byte is the rank: usable as the library's rank buffer
        template<typename range_t>
        inline constexpr bool ranks_in_place =
            std::ranges::contiguous_range<range_t> && sizeof(std::ranges::range_value_t<range_t>) == 1 &&
            std::is_trivially_copyable_v<std::ranges::range_value_t<range_t>>;

        template<typename range_t>
        std::vector<std::uint8_t> to_ranks(range_t const& r)
        {
            std::vector<std::uint8_t> out;
            if constexpr (std::ranges::sized_range<range_t>)
                out.reserve(std::ranges::size(r));
            for (auto const& c : r)
                out.push_back(static_cast<std::uint8_t>(c.to_rank()));
            return out;
        }
    }

    // result of search_batch(): CSR over the batch. offsets / status (and positions, for 32-bit position types) are views
    // of the library's result buffers, which this object keeps alive; copies of the object share them.
    template<typename position_t>
    struct kmer_batch_result
    {
        using positions_t = std::conditional_t<std::is_same_v<position_t, std::uint32_t>, detail::array_view<std::uint32_t>,
                                               std::vector<position_t>>;
        detail::array_view<std::uint64_t> offsets;   // [n_queries + 1]
        positions_t positions;                       // ascending per query
        detail::array_view<std::uint8_t> status;     // kmer_b200_query_status per query
        // approximate search with a hit strategy (empty otherwise): the Hamming distance of each position (same order),
        // when asked for, and d_min per query (0xFF without a hit) for every strategy but approx_hits::all()
        detail::array_view<std::uint8_t> distances;
        detail::array_view<std::uint8_t> best_distance;
        // seeding (seed_batch; empty otherwise): the query offset j of each position, and the occurrence count of every
        // k-mer of the batch (query order, then j order; max_occ + 1 for a k-mer above the cap)
        detail::array_view<std::uint32_t> seed_offsets;
        detail::array_view<std::uint32_t> kmer_counts;

        std::size_t size() const noexcept { return status.size(); }
        bool threw(std::size_t i) const { return status[i] == KMER_B200_QUERY_THROW_INVALID_ARGUMENT; }
        detail::kmer_index_result<position_t> operator[](std::size_t i) const
        {
            return detail::kmer_index_result<position_t>(
                std::vector<position_t>(positions.begin() + offsets[i], positions.begin() + offsets[i + 1]));
        }

        kmer_batch_result() = default;
        explicit kmer_batch_result(kmer_b200_result* r) : _owner(r, kmer_b200_result_free)
        {
            const std::uint64_t n_q = kmer_b200_result_n_queries(r), n_p = kmer_b200_result_n_positions(r);
            offsets = {kmer_b200_result_offsets(r), std::size_t(n_q + 1)};
            status = {kmer_b200_result_status(r), std::size_t(n_q)};
            if (kmer_b200_result_distances(r)) distances = {kmer_b200_result_distances(r), std::size_t(n_p)};
            if (kmer_b200_result_best_distances(r)) best_distance = {kmer_b200_result_best_distances(r), std::size_t(n_q)};
            if (kmer_b200_result_seed_offsets(r)) seed_offsets = {kmer_b200_result_seed_offsets(r), std::size_t(n_p)};
            if (kmer_b200_result_kmer_counts(r))
                kmer_counts = {kmer_b200_result_kmer_counts(r), std::size_t(kmer_b200_result_n_kmers(r))};
            if constexpr (std::is_same_v<position_t, std::uint32_t>)
                positions = {kmer_b200_result_positions(r), std::size_t(n_p)};
            else if (n_p)
                positions.assign(kmer_b200_result_positions(r), kmer_b200_result_positions(r) + n_p);
        }

    private:
        std::shared_ptr<kmer_b200_result> _owner;
    };

    // result of record_votes<k>(): per read, every (record, votes) with votes >= min_votes, by votes descending then record
    // ascending (CSR over the batch), and each read's counted k-mers. Views of the library's result buffers, which this
    // object keeps alive; copies of the object share them.
    struct record_votes_result
    {
        detail::array_view<std::uint64_t> offsets;    // [n_reads + 1]
        detail::array_view<std::uint32_t> records;    // record ids
        detail::array_view<std::uint32_t> votes;      // their votes
        detail::array_view<std::uint32_t> kmer_hits;  // [n_reads]
        detail::array_view<std::uint8_t> status;      // [n_reads], all KMER_B200_QUERY_OK

        std::size_t size() const noexcept { return status.size(); }
        // the (record, votes) pairs of read i
        std::vector<std::pair<std::uint32_t, std::uint32_t>> operator[](std::size_t i) const
        {
            std::vector<std::pair<std::uint32_t, std::uint32_t>> out;
            for (std::uint64_t e = offsets[i]; e < offsets[i + 1]; ++e) out.emplace_back(records[e], votes[e]);
            return out;
        }

        record_votes_result() = default;
        explicit record_votes_result(kmer_b200_result* r) : _owner(r, kmer_b200_result_free)
        {
            const std::uint64_t n_q = kmer_b200_result_n_queries(r), n_p = kmer_b200_result_n_positions(r);
            offsets = {kmer_b200_result_offsets(r), std::size_t(n_q + 1)};
            records = {kmer_b200_result_positions(r), std::size_t(n_p)};
            votes = {kmer_b200_result_votes(r), std::size_t(n_p)};
            kmer_hits = {kmer_b200_result_kmer_hits(r), std::size_t(n_q)};
            status = {kmer_b200_result_status(r), std::size_t(n_q)};
        }

    private:
        std::shared_ptr<kmer_b200_result> _owner;
    };

    // which hits of an approximate search (search_approx_batch): the seqan3 search_cfg::hit_all / hit_all_best /
    // hit_single_best / hit_strata{s} choices (kmer_b200_approx_hits)
    struct approx_hits
    {
        std::uint32_t strategy = KMER_B200_HITS_ALL;  // kmer_b200_approx_hits
        std::uint32_t s = 0;                          // strata(s) only

        static constexpr approx_hits all() noexcept { return {KMER_B200_HITS_ALL, 0}; }
        static constexpr approx_hits all_best() noexcept { return {KMER_B200_HITS_ALL_BEST, 0}; }
        static constexpr approx_hits single_best() noexcept { return {KMER_B200_HITS_SINGLE_BEST, 0}; }
        static constexpr approx_hits strata(std::uint32_t s) noexcept { return {KMER_B200_HITS_STRATA, s}; }
    };

    // tag for the shared-positions constructor below
    inline constexpr struct shared_positions_t {} shared_positions{};
    // tag for the collection constructor below
    inline constexpr struct collection_t {} collection{};

    // where a hit of a collection index lies: the text (record) and the offset inside it (kmer_index::locate)
    struct record_hit
    {
        std::uint32_t record = 0;
        std::uint32_t offset = 0;
        friend constexpr bool operator==(record_hit a, record_hit b) noexcept { return a.record == b.record && a.offset == b.offset; }
    };

    // kmer_index.hpp:350-566
    template<alphabet alphabet_t, typename position_t, std::size_t... ks>
    class kmer_index
    {
        static_assert(sizeof...(ks) > 0, "at least one k");
        static_assert(std::is_same_v<position_t, std::uint32_t>,
                      "the device index stores 32-bit positions (make_kmer_index fixes position_t = uint32_t, kmer_index.hpp:575)");
        // kmer_index.hpp:42-43
        static_assert(((ks > 0 && double(ks) < 64.0 / __builtin_log2(double(alphabet_size<alphabet_t>))) && ...),
                      "the hashspace for the current k cannot be represented with only a 64-bit integer. Please specify a valid k");

        using result_t = detail::kmer_index_result<position_t>;
        kmer_b200_index* _handle = nullptr;
        std::size_t _query_size_range = 10000;   // kmer_index.hpp:401

        explicit kmer_index(std::nullptr_t) {}   // empty shell for load()

    public:
        template<std::ranges::range text_t>
        explicit kmer_index(text_t& text, std::size_t /*n_threads*/ = 1, kmer_b200_mode mode = KMER_B200_MODE_REFERENCE_EXACT,
                            int device = -1)
        {
            build(text, mode, device, nullptr, 0);
        }

        // kmer_index(text, kmer::shared_positions): ONE position array, sorted by the largest k, serves every k (the
        // thesis' outlook, 04_outlook_and_conclusion.tex:25-45) -- about sizeof...(ks) times less device memory, the same
        // results, slower lookups through the shorter ks (KMER_B200_FLAG_SHARED_POSITIONS in kmer_b200.h)
        template<std::ranges::range text_t>
        kmer_index(text_t& text, shared_positions_t, kmer_b200_mode mode = KMER_B200_MODE_REFERENCE_EXACT, int device = -1)
        {
            build(text, mode, device, nullptr, 0, KMER_B200_FLAG_SHARED_POSITIONS);
        }

        // the same index replicated over several GPUs (built from key-range parts, one per GPU); search_batch() stripes
        // its batch over them
        template<std::ranges::range text_t>
        kmer_index(text_t& text, std::vector<int> const& devices, kmer_b200_mode mode = KMER_B200_MODE_REFERENCE_EXACT)
        {
            std::vector<std::int32_t> ids(devices.begin(), devices.end());
            build(text, mode, ids.empty() ? -1 : ids[0], ids.data(), std::uint32_t(ids.size()));
        }

        // kmer_index(texts, kmer::collection): one index over a collection of texts (a genome's chromosomes, a set of
        // transcripts), searched in CORRECT mode. No hit spans two texts: search_batch / search_approx_batch return what
        // searching each text on its own would, positions offset by the text's start in the concatenation; locate()
        // maps them to (text, offset) -- seqan3's (reference id, position) (kmer_b200_attach_records)
        template<std::ranges::range texts_t>
        kmer_index(texts_t const& texts, collection_t, int device = -1)
        {
            std::vector<std::uint8_t> ranks;
            std::vector<std::uint64_t> starts{0};
            gather_ranks(texts, ranks, starts);
            build(ranks, KMER_B200_MODE_CORRECT, device, nullptr, 0);
            detail::check(kmer_b200_attach_records(_handle, starts.data(), starts.size() - 1));
        }

        // (text, offset) of every position of a search result on a collection index, in the result's order; throws on an
        // index without texts
        std::vector<record_hit> locate(kmer_batch_result<position_t> const& result) const
        {
            const std::size_t n = result.positions.size();
            std::vector<std::uint32_t> rec(n), off(n);
            detail::check(kmer_b200_locate(_handle, result.positions.data(), n, rec.data(), off.data()));
            std::vector<record_hit> out(n);
            for (std::size_t i = 0; i < n; ++i) out[i] = record_hit{rec[i], off[i]};
            return out;
        }

    private:
        template<typename text_t>
        void build(text_t& text, kmer_b200_mode mode, int device, std::int32_t const* ids, std::uint32_t n_ids,
                   std::uint32_t flags = 0)
        {
            static constexpr std::uint32_t k_list[] = {std::uint32_t(ks)...};
            kmer_b200_config cfg;
            kmer_b200_config_default(&cfg);
            cfg.mode = mode;
            cfg.device = device;
            cfg.reserved = flags;
            if (n_ids > 1)
            {
                cfg.device_ids = ids;
                cfg.n_devices = n_ids;
            }
            if constexpr (detail::ranks_in_place<text_t>)
            {
                // std::vector<alphabet_t> of 1-byte alphabet objects: the storage is the rank array
                detail::check(kmer_b200_create(reinterpret_cast<std::uint8_t const*>(std::ranges::data(text)), std::ranges::size(text),
                                               std::uint32_t(alphabet_size<alphabet_t>), k_list, sizeof...(ks), &cfg, &_handle));
            }
            else
            {
                auto ranks = detail::to_ranks(text);
                detail::check(kmer_b200_create(ranks.data(), ranks.size(), std::uint32_t(alphabet_size<alphabet_t>), k_list,
                                               sizeof...(ks), &cfg, &_handle));
            }
        }

    public:
        // construct once, load later: kmer_index<...>::load(path) restores an index written by save(path)
        void save(std::string const& path) const { detail::check(kmer_b200_save(_handle, path.c_str())); }
        static kmer_index load(std::string const& path, kmer_b200_mode mode = KMER_B200_MODE_REFERENCE_EXACT, int device = -1)
        {
            kmer_b200_config cfg;
            kmer_b200_config_default(&cfg);
            cfg.mode = mode;
            cfg.device = device;
            kmer_index out{nullptr};
            detail::check(kmer_b200_load(path.c_str(), &cfg, &out._handle));
            static constexpr std::uint32_t k_list[] = {std::uint32_t(ks)...};
            if (kmer_b200_n_elements(out._handle) != sizeof...(ks))
                throw std::invalid_argument("index file holds a different set of ks");
            for (std::uint32_t i = 0; i < sizeof...(ks); ++i)
            {
                kmer_b200_element_info info;
                detail::check(kmer_b200_element_info_get(out._handle, i, &info));
                if (info.k != k_list[i])
                    throw std::invalid_argument("index file holds a different set of ks");
            }
            return out;
        }

        kmer_index(kmer_index const&) = delete;
        kmer_index& operator=(kmer_index const&) = delete;
        kmer_index(kmer_index&& o) noexcept : _handle(std::exchange(o._handle, nullptr)), _query_size_range(o._query_size_range) {}
        kmer_index& operator=(kmer_index&& o) noexcept
        {
            if (this != &o)
            {
                kmer_b200_destroy(_handle);
                _handle = std::exchange(o._handle, nullptr);
            }
            return *this;
        }
        ~kmer_index() { kmer_b200_destroy(_handle); }

        // kmer_index.hpp:498-502: the scheme table is built for query lengths below 10000
        void extend_query_size_range(std::size_t new_maximum)
        {
            if (new_maximum > 10000)
                throw std::invalid_argument("query size range above 10000 is not supported");
        }

        // All queries in one launch. queries: any range of ranges of alphabet_t.
        template<std::ranges::range queries_t>
        kmer_batch_result<position_t> search_batch(queries_t const& queries) const
        {
            using query_t = std::remove_cvref_t<std::ranges::range_reference_t<queries_t const>>;
            kmer_b200_result* r = nullptr;
            if constexpr (detail::ranks_in_place<query_t> && std::is_lvalue_reference_v<std::ranges::range_reference_t<queries_t const>>)
            {
                // queries in their own contiguous 1-byte storage: hand over pointers, the library gathers them in parallel
                if constexpr (std::ranges::random_access_range<queries_t const> && std::ranges::sized_range<queries_t const>)
                {
                    // (a batch of 10^8 std::vectors: collecting the pointers is 2.4 GB of reads -- all cores)
                    const std::size_t n_q = std::ranges::size(queries);
                    std::unique_ptr<std::uint8_t const*[]> ptrs(new std::uint8_t const*[n_q]);
                    std::unique_ptr<std::uint64_t[]> lens(new std::uint64_t[n_q]);
                    detail::parallel_ranges(n_q, [&](std::size_t lo, std::size_t hi) {
                        auto it = std::ranges::begin(queries) + static_cast<std::ranges::range_difference_t<queries_t const>>(lo);
                        for (std::size_t i = lo; i < hi; ++i, ++it)
                        {
                            ptrs[i] = reinterpret_cast<std::uint8_t const*>(std::ranges::data(*it));
                            lens[i] = std::ranges::size(*it);
                        }
                    });
                    detail::check(kmer_b200_search_batch_ptrs(_handle, ptrs.get(), lens.get(), n_q, UINT32_MAX, &r));
                }
                else
                {
                    std::vector<std::uint8_t const*> ptrs;
                    std::vector<std::uint64_t> lens;
                    for (auto const& q : queries)
                    {
                        ptrs.push_back(reinterpret_cast<std::uint8_t const*>(std::ranges::data(q)));
                        lens.push_back(std::ranges::size(q));
                    }
                    detail::check(kmer_b200_search_batch_ptrs(_handle, ptrs.data(), lens.data(), ptrs.size(), UINT32_MAX, &r));
                }
            }
            else
            {
                std::vector<std::uint8_t> ranks;
                std::vector<std::uint64_t> offsets{0};
                for (auto const& q : queries)
                {
                    for (auto const& c : q)
                        ranks.push_back(static_cast<std::uint8_t>(c.to_rank()));
                    offsets.push_back(ranks.size());
                }
                detail::check(kmer_b200_search_batch(_handle, ranks.data(), offsets.data(), offsets.size() - 1, UINT32_MAX, &r));
            }
            return kmer_batch_result<position_t>(r);
        }

        // Approximate search (no reference analogue; kmer_b200_search_approx_batch): per query, every position whose window
        // differs from the query in at most max_mismatches (<= 8) symbols, ascending. Substitutions only; max_mismatches = 0
        // is exact search in CORRECT mode. The batch is gathered into one rank buffer (a copy of the bytes when the queries
        // hold their ranks in place) and staged on the device in one copy.
        template<std::ranges::range queries_t>
        kmer_batch_result<position_t> search_approx_batch(queries_t const& queries, std::uint32_t max_mismatches) const
        {
            std::vector<std::uint8_t> ranks;
            std::vector<std::uint64_t> offsets{0};
            gather_ranks(queries, ranks, offsets);
            kmer_b200_result* r = nullptr;
            detail::check(kmer_b200_search_approx_batch(_handle, ranks.data(), offsets.data(), offsets.size() - 1, max_mismatches, &r));
            return kmer_batch_result<position_t>(r);
        }

        // Approximate search with a hit strategy (kmer_b200_search_approx_batch_ex): approx_hits::all() (every hit),
        // all_best() (the hits at the smallest distance d_min), single_best() (the lowest such position) or strata(s)
        // (distance <= min(max_mismatches, d_min + s)). The result's best_distance holds d_min per query (not for all()),
        // and `distances` the Hamming distance of every position when asked for.
        template<std::ranges::range queries_t>
        kmer_batch_result<position_t> search_approx_batch(queries_t const& queries, std::uint32_t max_mismatches, approx_hits hits,
                                                          bool distances = false) const
        {
            std::vector<std::uint8_t> ranks;
            std::vector<std::uint64_t> offsets{0};
            gather_ranks(queries, ranks, offsets);
            kmer_b200_approx_options opt{max_mismatches, hits.strategy, hits.s, distances ? std::uint32_t(KMER_B200_APPROX_DISTANCES) : 0u};
            kmer_b200_result* r = nullptr;
            detail::check(kmer_b200_search_approx_batch_ex(_handle, ranks.data(), offsets.data(), offsets.size() - 1, &opt, &r));
            return kmer_batch_result<position_t>(r);
        }

        // k-mer seeding (kmer_b200_seed_batch; search_k<k> for every offset of every query in one call): per query, for
        // every offset j in [0, m - k], every position p of the k-mer q[j, j+k), ordered by (j, p), with j in
        // seed_offsets and each k-mer's occurrence count in kmer_counts. max_occ > 0: k-mers occurring more often give no
        // positions and count max_occ + 1. On a collection index only windows inside one record count.
        template<std::size_t k, std::ranges::range queries_t>
        kmer_batch_result<position_t> seed_batch(queries_t const& queries, std::uint32_t max_occ = 0) const
        {
            static_assert(((k == ks) || ...), "seed_batch<k>: k is not one of this index's ks");
            std::vector<std::uint8_t> ranks;
            std::vector<std::uint64_t> offsets{0};
            gather_ranks(queries, ranks, offsets);
            kmer_b200_result* r = nullptr;
            detail::check(kmer_b200_seed_batch(_handle, ranks.data(), offsets.data(), offsets.size() - 1, std::uint32_t(k), max_occ, &r));
            return kmer_batch_result<position_t>(r);
        }

        // record votes on a collection index (kmer_b200_record_votes; attach_records first): per read, every record r that
        // at least min_votes of its counted k-mers occur in (1 <= in-record occurrences, <= max_occ when max_occ > 0; a
        // k-mer gives each record it occurs in one vote), by votes descending then record ascending
        template<std::size_t k, std::ranges::range queries_t>
        record_votes_result record_votes(queries_t const& queries, std::uint32_t max_occ = 0, std::uint32_t min_votes = 1) const
        {
            static_assert(((k == ks) || ...), "record_votes<k>: k is not one of this index's ks");
            std::vector<std::uint8_t> ranks;
            std::vector<std::uint64_t> offsets{0};
            gather_ranks(queries, ranks, offsets);
            kmer_b200_result* r = nullptr;
            detail::check(kmer_b200_record_votes(_handle, ranks.data(), offsets.data(), offsets.size() - 1, std::uint32_t(k), max_occ,
                                                 min_votes, &r));
            return record_votes_result(r);
        }

        // k-mer spectrum of element k (kmer_b200_spectrum): hist[c] = distinct k-mers occurring c times for
        // 1 <= c < bins - 1, hist[bins - 1] = those occurring bins - 1 times or more, hist[0] = sigma^k - distinct. On a
        // collection index only windows inside one record count.
        struct kmer_spectrum
        {
            std::vector<std::uint64_t> hist;
            kmer_b200_spectrum_info info{};
        };
        template<std::size_t k>
        kmer_spectrum spectrum(std::uint64_t bins = 10001) const
        {
            static_assert(((k == ks) || ...), "spectrum<k>: k is not one of this index's ks");
            kmer_spectrum s;
            s.hist.resize(bins);
            detail::check(kmer_b200_spectrum(_handle, std::uint32_t(k), s.hist.data(), bins, &s.info));
            return s;
        }

        // the k-mers occurring at least min_count times as (hash, count), count descending then hash ascending, the
        // first cap of them (kmer_b200_frequent_kmers)
        template<std::size_t k>
        std::vector<std::pair<std::uint64_t, std::uint64_t>> frequent_kmers(std::uint64_t min_count, std::uint64_t cap) const
        {
            static_assert(((k == ks) || ...), "frequent_kmers<k>: k is not one of this index's ks");
            std::vector<std::uint64_t> hashes(cap), counts(cap);
            std::uint64_t n = 0;
            detail::check(kmer_b200_frequent_kmers(_handle, std::uint32_t(k), min_count, hashes.data(), counts.data(), cap, &n));
            std::vector<std::pair<std::uint64_t, std::uint64_t>> out(std::min(n, cap));
            for (std::size_t i = 0; i < out.size(); ++i) out[i] = {hashes[i], counts[i]};
            return out;
        }

        // the repeat cap that ignores the most frequent `fraction` of the distinct k-mers (kmer_b200_occurrence_cutoff);
        // seed_batch<k>(queries, cutoff) drops exactly the k-mers above it
        template<std::size_t k>
        std::uint64_t occurrence_cutoff(double fraction) const
        {
            static_assert(((k == ks) || ...), "occurrence_cutoff<k>: k is not one of this index's ks");
            std::uint64_t c = 0;
            detail::check(kmer_b200_occurrence_cutoff(_handle, std::uint32_t(k), fraction, &c));
            return c;
        }

        // one query: its positions within max_mismatches substitutions, ascending; throws for an empty query
        std::vector<position_t> search_approx(std::vector<alphabet_t> const& query, std::uint32_t max_mismatches) const
        {
            std::array<std::vector<alphabet_t> const*, 1> one{&query};
            auto deref = one | std::views::transform([](auto const* p) -> std::vector<alphabet_t> const& { return *p; });
            auto batch = search_approx_batch(deref, max_mismatches);
            if (batch.status[0] != KMER_B200_QUERY_OK)
                throw std::invalid_argument("approximate search of an empty query is undefined");
            return std::vector<position_t>(batch.positions.begin(), batch.positions.end());
        }

    private:
        // a batch as one rank buffer and its offsets (a copy of the bytes when the queries hold their ranks in place)
        template<std::ranges::range queries_t>
        static void gather_ranks(queries_t const& queries, std::vector<std::uint8_t>& ranks, std::vector<std::uint64_t>& offsets)
        {
            using query_t = std::remove_cvref_t<std::ranges::range_reference_t<queries_t const>>;
            for (auto const& q : queries)
            {
                if constexpr (detail::ranks_in_place<query_t>)
                {
                    auto const* p = reinterpret_cast<std::uint8_t const*>(std::ranges::data(q));
                    ranks.insert(ranks.end(), p, p + std::ranges::size(q));
                }
                else
                {
                    for (auto const& c : q)
                        ranks.push_back(static_cast<std::uint8_t>(c.to_rank()));
                }
                offsets.push_back(ranks.size());
            }
        }

    public:

        // kmer_index_element::search_k (kmer_index.hpp:182-190): the bucket of the k symbols starting at `it`, for one
        // of the index's ks; empty when the k-mer does not occur (the reference returns a null pointer)
        template<std::size_t k, typename iterator_t>
        result_t search_k(iterator_t it) const
        {
            static_assert(((k == ks) || ...), "search_k<k>: k is not one of this index's ks");
            std::vector<alphabet_t> kmer_symbols;
            for (std::size_t i = 0; i < k; ++i, ++it) kmer_symbols.push_back(*it);
            return search(kmer_symbols);
        }

        // kmer_index.hpp:505-558. A batch of one: correct, but a GPU is fed with search_batch().
        result_t search(std::vector<alphabet_t>& query) const
        {
            if (query.size() > _query_size_range)   // :507-509
                throw std::invalid_argument("query size exceed the maximum size " + std::to_string(_query_size_range) + " specified");
            std::array<std::vector<alphabet_t> const*, 1> one{&query};
            auto deref = one | std::views::transform([](auto const* p) -> std::vector<alphabet_t> const& { return *p; });
            auto batch = search_batch(deref);
            if (batch.status[0] == KMER_B200_QUERY_THROW_INVALID_ARGUMENT)   // :119-122
                throw std::invalid_argument("query size too low for specified k");
            if (batch.status[0] != KMER_B200_QUERY_OK)
                throw std::invalid_argument("query length 0 or 10000 is undefined in the reference (kmer_index.hpp:195,512)");
            return result_t(std::vector<position_t>(batch.positions.begin(), batch.positions.end()));
        }

        result_t search(std::vector<alphabet_t>&& query) const   // :561-565, with the missing return
        {
            auto hold = std::move(query);
            return search(hold);
        }

        kmer_b200_index* native_handle() const noexcept { return _handle; }
    };

    // kmer_index.hpp:569-579
    template<std::size_t... ks, std::ranges::range text_t>
    auto make_kmer_index(text_t&& text, std::size_t n_threads = 1)
    {
        using alphabet_t = std::ranges::range_value_t<std::remove_cvref_t<text_t>>;
        using position_t = std::uint32_t;
        return kmer_index<alphabet_t, position_t, ks...>(text, n_threads);
    }

    // names used by the thesis (thesis/content/02_implementation.tex:253-274)
    template<typename alphabet_t, std::size_t k>
    using single_kmer_index = kmer_index<alphabet_t, std::uint32_t, k>;
    template<typename alphabet_t, std::size_t... ks>
    using multi_kmer_index = kmer_index<alphabet_t, std::uint32_t, ks...>;
}   // namespace kmer
