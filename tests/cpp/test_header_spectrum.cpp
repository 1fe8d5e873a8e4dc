// k-mer spectrum through include/kmer_index.hpp: spectrum<k>, frequent_kmers<k> and occurrence_cutoff<k> against a plain
// std::map count of every window, on a random dna4 text with one long repeat. Exit code 0 = all good. Needs a GPU at run
// time; compile-only is part of the CPU test suite.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <vector>

#include <kmer_index.hpp>

using alphabet_t = kmer::dna4;

static uint64_t lcg_state = 0x2545F4914F6CDD1Dull;
static uint32_t next_u32()
{
    lcg_state = lcg_state * 6364136223846793005ull + 1442695040888963407ull;
    return uint32_t(lcg_state >> 33);
}

#define REQUIRE(cond)                                                        \
    do {                                                                     \
        if (!(cond)) {                                                       \
            std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); \
            return 1;                                                        \
        }                                                                    \
    } while (0)

template<size_t k>
static std::map<uint64_t, uint64_t> brute_counts(std::vector<alphabet_t> const& text)
{
    std::map<uint64_t, uint64_t> c;
    for (size_t p = 0; p + k <= text.size(); ++p)
    {
        uint64_t h = 0;
        for (size_t i = 0; i < k; ++i) h = h * 4 + text[p + i].to_rank();
        ++c[h];
    }
    return c;
}

template<size_t k, typename index_t>
static int check_k(index_t const& ix, std::vector<alphabet_t> const& text)
{
    const auto want = brute_counts<k>(text);
    for (uint64_t bins : {2ull, 7ull, 100ull})
    {
        auto s = ix.template spectrum<k>(bins);
        std::vector<uint64_t> hist(bins, 0);
        uint64_t mx = 0;
        for (auto const& [h, c] : want)
        {
            ++hist[std::min<uint64_t>(c, bins - 1)];
            mx = std::max(mx, c);
        }
        hist[0] = (uint64_t(1) << (2 * k)) - want.size();
        REQUIRE(s.hist == hist);
        REQUIRE(s.info.total == text.size() - k + 1);
        REQUIRE(s.info.distinct == want.size());
        REQUIRE(s.info.max_count == mx);
        REQUIRE(s.info.key_space == (uint64_t(1) << (2 * k)));
    }
    std::vector<std::pair<uint64_t, uint64_t>> order;
    for (auto const& [h, c] : want) order.push_back({h, c});
    std::stable_sort(order.begin(), order.end(), [](auto const& a, auto const& b) { return a.second > b.second; });
    auto top = ix.template frequent_kmers<k>(1, 25);
    REQUIRE(top.size() == 25);
    for (size_t i = 0; i < top.size(); ++i) REQUIRE(top[i] == order[i]);
    for (double f : {0.0, 0.001, 0.5})
    {
        const uint64_t F = uint64_t(std::floor(f * double(want.size())));
        uint64_t cut = 1;
        while (true)
        {
            uint64_t above = 0;
            for (auto const& [h, c] : want) above += c > cut;
            if (above <= F) break;
            ++cut;
        }
        REQUIRE(ix.template occurrence_cutoff<k>(f) == cut);
    }
    return 0;
}

int main()
{
    std::vector<alphabet_t> text(60000);
    for (auto& c : text) c.assign_rank(uint8_t(next_u32() % 4));
    for (size_t p = 30000; p < 33000; ++p) text[p].assign_rank(uint8_t(p % 3 == 0));  // a period-3 repeat
    kmer::kmer_index<alphabet_t, uint32_t, 6, 12> ix(text, 1, KMER_B200_MODE_CORRECT);
    if (check_k<6>(ix, text)) return 1;
    if (check_k<12>(ix, text)) return 1;
    std::printf("all checks passed\n");
    return 0;
}
