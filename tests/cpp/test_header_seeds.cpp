// k-mer seeding through include/kmer_index.hpp: seed_batch<k> on a std::vector<std::vector<dna4>> equals search_k<k> at
// every offset of every query, with the cap and the per-k-mer counts, and reads across a record start of a collection get
// only in-record hits. Exit code 0 = all good. Needs a GPU at run time; compile-only is part of the CPU test suite.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include <kmer_index.hpp>

using alphabet_t = kmer::dna4;

static uint64_t lcg_state = 0x9E3779B97F4A7C15ull;
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
    for (size_t p = 20000; p < 23000; ++p) text[p].assign_rank(0);   // a repeat: one 10-mer with ~3000 positions
    kmer::kmer_index<alphabet_t, uint32_t, 10, 12> ix(text, 1, KMER_B200_MODE_CORRECT);

    std::vector<std::vector<alphabet_t>> queries;
    for (int i = 0; i < 200; ++i)
    {
        size_t m = next_u32() % 160;
        if (i % 2 == 0 && m <= text.size())
        {
            size_t s = i % 10 == 0 ? 21000 : next_u32() % (text.size() - m + 1);
            queries.emplace_back(text.begin() + s, text.begin() + s + m);
        }
        else
            queries.push_back(random_sequence(m));
    }
    for (uint32_t max_occ : {0u, 50u})
    {
        auto res = ix.seed_batch<10>(queries, max_occ);
        REQUIRE(res.size() == queries.size());
        size_t kmer = 0;
        for (size_t i = 0; i < queries.size(); ++i)
        {
            REQUIRE(res.status[i] == KMER_B200_QUERY_OK);
            size_t at = res.offsets[i];
            for (size_t j = 0; j + 10 <= queries[i].size(); ++j, ++kmer)
            {
                auto want = ix.search_k<10>(queries[i].begin() + j).to_vector();
                const bool capped = max_occ && want.size() > max_occ;
                REQUIRE(res.kmer_counts[kmer] == (capped ? max_occ + 1 : want.size()));
                if (capped) continue;
                for (auto p : want)
                {
                    REQUIRE(at < res.offsets[i + 1]);
                    REQUIRE(res.positions[at] == p && res.seed_offsets[at] == j);
                    ++at;
                }
            }
            REQUIRE(at == res.offsets[i + 1]);
        }
        REQUIRE(kmer == res.kmer_counts.size());
    }

    // a collection of two texts: a read across their junction has no hit spanning it
    std::vector<std::vector<alphabet_t>> texts{random_sequence(5000), random_sequence(7000)};
    kmer::kmer_index<alphabet_t, uint32_t, 12> coll(texts, kmer::collection);
    std::vector<alphabet_t> read(texts[0].end() - 30, texts[0].end());
    read.insert(read.end(), texts[1].begin(), texts[1].begin() + 30);
    auto r = coll.seed_batch<12>(std::vector<std::vector<alphabet_t>>{read});
    for (size_t h = 0; h < r.positions.size(); ++h)
        REQUIRE(r.positions[h] + 12 <= 5000 || r.positions[h] >= 5000);
    REQUIRE(r.kmer_counts.size() == 60 - 12 + 1);
    for (size_t j = 19; j < 30; ++j) REQUIRE(r.kmer_counts[j] == 0 || r.kmer_counts[j] < 3);   // junction 12-mers: random elsewhere

    std::printf("all checks passed\n");
    return 0;
}
