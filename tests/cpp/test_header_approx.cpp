// Approximate search through include/kmer_index.hpp: search_approx_batch on a std::vector<std::vector<dna4>> equals
// search_approx per query and a plain Hamming scan, and with 0 mismatches equals search_batch of a CORRECT-mode index.
// Exit code 0 = all good. Needs a GPU at run time; compile-only is part of the CPU test suite.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include <kmer_index.hpp>

using alphabet_t = kmer::dna4;

static uint64_t lcg_state = 0x2545F4914F6CDD1Dull;
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

static std::vector<uint32_t> hamming_scan(std::vector<alphabet_t> const& text, std::vector<alphabet_t> const& q, uint32_t e)
{
    std::vector<uint32_t> out;
    if (q.empty() || q.size() > text.size()) return out;
    for (size_t p = 0; p + q.size() <= text.size(); ++p)
    {
        uint32_t d = 0;
        for (size_t i = 0; i < q.size() && d <= e; ++i) d += text[p + i] != q[i];
        if (d <= e) out.push_back(uint32_t(p));
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

int main()
{
    auto text = random_sequence(100000);
    kmer::kmer_index<alphabet_t, uint32_t, 12> ix(text, 1, KMER_B200_MODE_CORRECT);

    // text windows (some at 0 and ending at n) with up to 3 substitutions, plus random reads; lengths 1..120
    std::vector<std::vector<alphabet_t>> queries;
    for (int i = 0; i < 300; ++i)
    {
        size_t m = 1 + next_u32() % 120;
        if (i % 3 == 2)
        {
            queries.push_back(random_sequence(m));
            continue;
        }
        size_t start = i % 11 == 0 ? 0 : (i % 11 == 1 ? text.size() - m : next_u32() % (text.size() - m + 1));
        std::vector<alphabet_t> q(text.begin() + start, text.begin() + start + m);
        for (int s = 0, d = i % 4; s < d; ++s) q[next_u32() % m].assign_rank(uint8_t(next_u32() % 4));
        queries.push_back(std::move(q));
    }

    for (uint32_t e : {0u, 1u, 3u})
    {
        auto batch = ix.search_approx_batch(queries, e);
        REQUIRE(batch.size() == queries.size());
        for (size_t i = 0; i < queries.size(); ++i)
        {
            std::vector<uint32_t> got(batch.positions.begin() + batch.offsets[i], batch.positions.begin() + batch.offsets[i + 1]);
            REQUIRE(got == ix.search_approx(queries[i], e));
            REQUIRE(got == hamming_scan(text, queries[i], e));
        }
        if (e == 0)
        {
            auto exact = ix.search_batch(queries);
            REQUIRE(exact.offsets.size() == batch.offsets.size());
            for (size_t i = 0; i <= queries.size(); ++i) REQUIRE(exact.offsets[i] == batch.offsets[i]);
            for (size_t i = 0; i < batch.positions.size(); ++i) REQUIRE(exact.positions[i] == batch.positions[i]);
        }
    }
    bool threw = false;
    try
    {
        ix.search_approx(queries[0], 9);
    }
    catch (std::invalid_argument const&)
    {
        threw = true;
    }
    REQUIRE(threw);
    std::printf("all checks passed\n");
    return 0;
}
