// Exercises include/kmer_index.hpp the way a user of the reference would (test_main.cpp:21-69 protocol):
// build single and multi indices with make_kmer_index, search(), compare to_vector() with a plain scan.
// Exit code 0 = all good. Needs a GPU at run time; compile-only is part of the CPU test suite.
// argv[1]: directory for the save / load round trip (default: the system's temporary directory).
#include <cstdio>
#include <cstdlib>
#include <filesystem>
#include <string>
#include <vector>

#include <kmer_index.hpp>

using alphabet_t = kmer::dna4;

static uint64_t lcg_state = 88172645463325252ull;
static uint32_t next_u32()
{
    lcg_state = lcg_state * 6364136223846793005ull + 1442695040888963407ull;
    return uint32_t(lcg_state >> 33);
}

static std::vector<alphabet_t> random_sequence(size_t n)
{
    std::vector<alphabet_t> s(n);
    for (auto& c : s) c.assign_rank(uint8_t(next_u32() % 4));
    return s;
}

static std::vector<uint32_t> scan(std::vector<alphabet_t> const& text, std::vector<alphabet_t> const& q)
{
    std::vector<uint32_t> out;
    if (q.size() > text.size()) return out;
    for (size_t p = 0; p + q.size() <= text.size(); ++p)
    {
        bool eq = true;
        for (size_t i = 0; i < q.size() && eq; ++i) eq = text[p + i] == q[i];
        if (eq) out.push_back(uint32_t(p));
    }
    return out;
}

#define REQUIRE(cond)                                                        \
    do {                                                                     \
        if (!(cond)) {                                                       \
            std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); \
            return 1;                                                        \
        }                                                                    \
    } while (0)

int main(int argc, char** argv)
{
    static_assert(kmer::detail::fast_pow(4, 12) == 16777216);
    static_assert(kmer::detail::fast_pow(2, 63) == 0 && kmer::detail::fast_pow(1, 200) == 1);

    auto text = random_sequence(200000);
    auto single = kmer::make_kmer_index<10>(text);
    auto multi = kmer::make_kmer_index<10, 11, 12>(text);
    kmer::single_kmer_index<alphabet_t, 16> k16(text);

    // lengths on which the reference is correct for these indices: k-5 .. 2k-1 (test_main.cpp:32)
    for (size_t m = 5; m < 20; ++m)
        for (int rep = 0; rep < 6; ++rep)
        {
            std::vector<alphabet_t> q;
            if (rep % 2 == 0) {
                size_t start = next_u32() % (text.size() - m + 1);
                if (rep == 4) start = text.size() - m;   // ends at the end of the text
                q.assign(text.begin() + start, text.begin() + start + m);
            } else {
                q = random_sequence(m);
            }
            auto truth = scan(text, q);
            REQUIRE(single.search(q).to_vector() == truth);
            REQUIRE(multi.search(q).to_vector() == truth);
            REQUIRE(single.search(q).size() == truth.size());
        }

    // rvalue overload returns (the reference's does not)
    {
        std::vector<alphabet_t> q(text.begin() + 77, text.begin() + 87);
        REQUIRE(single.search(std::vector<alphabet_t>(q)).to_vector() == scan(text, q));
    }
    // the reference throws std::invalid_argument when the rest is too short for k (kmer_index.hpp:119-122):
    // k = 16, m = 17 -> rest 1 -> 4^15 > 1e7, once the full part is present
    {
        std::vector<alphabet_t> q(text.begin() + 1000, text.begin() + 1017);
        bool threw = false;
        try { (void)k16.search(q); } catch (std::invalid_argument const&) { threw = true; }
        REQUIRE(threw);
        std::vector<alphabet_t> too_long(10001);
        threw = false;
        try { (void)k16.search(too_long); } catch (std::invalid_argument const&) { threw = true; }
        REQUIRE(threw);
    }
    // batch API
    {
        std::vector<std::vector<alphabet_t>> qs;
        for (int i = 0; i < 100; ++i) {
            size_t m = 10 + i % 10, start = next_u32() % (text.size() - m + 1);
            qs.emplace_back(text.begin() + start, text.begin() + start + m);
        }
        auto batch = single.search_batch(qs);
        REQUIRE(batch.size() == qs.size());
        for (size_t i = 0; i < qs.size(); ++i)
            REQUIRE(batch[i].to_vector() == scan(text, qs[i]));
    }
    // the reference's result surface (kmer_index_result.hpp:203-270): bucket + mask, should_use / should_not_use
    {
        std::vector<uint32_t> bucket{40, 10, 30, 20};
        kmer::detail::kmer_index_result<uint32_t> r(&bucket, false);
        REQUIRE(r.size() == 0 && r.to_vector().empty());
        r.should_use(0);
        r.should_use(3);
        REQUIRE((r.to_vector() == std::vector<uint32_t>{20, 40}));
        r.should_not_use(0);
        REQUIRE((r.to_vector() == std::vector<uint32_t>{20}));
        std::vector<uint32_t> other{5};
        std::vector<std::vector<uint32_t> const*> buckets{&bucket, &other};
        kmer::detail::kmer_index_result<uint32_t> many(buckets);
        REQUIRE((many.to_vector() == std::vector<uint32_t>{5, 10, 20, 30, 40}));
        // element-level exact lookup from an iterator (kmer_index.hpp:182-190)
        REQUIRE(single.search_k<10>(text.begin() + 321).to_vector() ==
                scan(text, std::vector<alphabet_t>(text.begin() + 321, text.begin() + 331)));
        REQUIRE(multi.search_k<11>(text.begin() + 99).to_vector() ==
                scan(text, std::vector<alphabet_t>(text.begin() + 99, text.begin() + 110)));
    }
    // one index over all the GPUs of the box (kmer_b200_config.device_ids): same answers as the one-device index
    {
        int n_dev = 0;
        if (std::getenv("KMER_B200_TEST_DEVICES")) n_dev = std::atoi(std::getenv("KMER_B200_TEST_DEVICES"));
        if (n_dev >= 2)
        {
            std::vector<int> devices;
            for (int d = 0; d < n_dev; ++d) devices.push_back(d);
            kmer::kmer_index<alphabet_t, uint32_t, 10, 11, 12> wide(text, devices);
            std::vector<std::vector<alphabet_t>> qs;
            for (int i = 0; i < 2000; ++i) {
                size_t m = 5 + i % 15, start = next_u32() % (text.size() - m + 1);
                qs.emplace_back(text.begin() + start, text.begin() + start + m);
            }
            auto a = wide.search_batch(qs), b = multi.search_batch(qs);
            REQUIRE(a.offsets == b.offsets && a.positions == b.positions && a.status == b.status);
            std::printf("multi-device index over %d GPUs: ok\n", n_dev);
        }
    }
    // shared-positions index (one position array for all ks): the same answers, also at the end of the text
    {
        kmer::kmer_index<alphabet_t, uint32_t, 10, 11, 12> shared(text, kmer::shared_positions);
        std::vector<std::vector<alphabet_t>> qs;
        for (int i = 0; i < 2000; ++i) {
            size_t m = 5 + i % 30, start = next_u32() % (text.size() - m + 1);
            qs.emplace_back(text.begin() + start, text.begin() + start + m);
        }
        for (size_t m = 5; m < 30; ++m) qs.emplace_back(text.end() - m, text.end());
        auto a = shared.search_batch(qs), b = multi.search_batch(qs);
        REQUIRE(a.offsets == b.offsets && a.positions == b.positions && a.status == b.status);
    }
    // other alphabets
    {
        std::vector<kmer::dna15> t15(50000);
        for (auto& c : t15) c.assign_rank(uint8_t(next_u32() % 15));
        auto idx = kmer::make_kmer_index<8>(t15);
        std::vector<kmer::dna15> q(t15.begin() + 123, t15.begin() + 131);
        auto r = idx.search(q).to_vector();
        REQUIRE(!r.empty() && r.front() <= 123);
    }
    // save / load round trip
    {
        const std::string path =
            ((argc > 1 ? std::filesystem::path(argv[1]) : std::filesystem::temp_directory_path()) / "kmer_index_hpp_test.kmerb200").string();
        multi.save(path);
        auto loaded = kmer::kmer_index<alphabet_t, uint32_t, 10, 11, 12>::load(path);
        std::vector<alphabet_t> q(text.begin() + 4242, text.begin() + 4242 + 17);
        REQUIRE(loaded.search(q).to_vector() == multi.search(q).to_vector());
        bool threw = false;
        try { (void)kmer::kmer_index<alphabet_t, uint32_t, 10>::load(path); } catch (std::invalid_argument const&) { threw = true; }
        REQUIRE(threw);
        std::remove(path.c_str());
    }
    std::printf("kmer_index.hpp: all checks passed\n");
    return 0;
}
