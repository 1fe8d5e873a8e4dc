// Record votes through include/kmer_index.hpp: record_votes<k> on a collection of texts equals a std::map tally of, for
// every k-mer of every read, the texts it occurs in (inside one text), with the cap and min_votes, ordered by votes
// descending then text ascending. Exit code 0 = all good. Needs a GPU at run time; compile-only is part of the CPU suite.
#include <algorithm>
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

constexpr size_t k = 12;

// occurrences of q[j, j + k) inside text t
static uint32_t occurrences(std::vector<alphabet_t> const& t, std::vector<alphabet_t> const& q, size_t j)
{
    uint32_t c = 0;
    for (size_t p = 0; p + k <= t.size(); ++p)
    {
        bool eq = true;
        for (size_t i = 0; i < k && eq; ++i) eq = t[p + i] == q[j + i];
        c += eq;
    }
    return c;
}

int main()
{
    // 60 texts: random ones, near-copies of a shared one (so k-mers vote for several texts), an empty one and a short one
    auto base = random_sequence(3000);
    std::vector<std::vector<alphabet_t>> texts;
    for (int t = 0; t < 60; ++t)
    {
        if (t == 7) texts.emplace_back();
        else if (t == 8) texts.push_back(random_sequence(k));
        else if (t % 3 == 0)
        {
            auto c = base;
            for (int s = 0; s < 30; ++s) c[next_u32() % c.size()].assign_rank(uint8_t(next_u32() % 4));
            texts.push_back(c);
        }
        else texts.push_back(random_sequence(500 + next_u32() % 2000));
    }
    kmer::kmer_index<alphabet_t, uint32_t, 12> coll(texts, kmer::collection);

    std::vector<std::vector<alphabet_t>> reads;
    for (int i = 0; i < 60; ++i)
    {
        auto const& t = texts[next_u32() % texts.size()];
        size_t m = 5 + next_u32() % 150;
        if (i % 4 == 3 || t.size() < m) reads.push_back(random_sequence(m));
        else
        {
            size_t s = next_u32() % (t.size() - m + 1);
            reads.emplace_back(t.begin() + s, t.begin() + s + m);
        }
    }
    for (uint32_t max_occ : {0u, 3u, 25u})
        for (uint32_t min_votes : {1u, 2u, 40u})
        {
            auto res = coll.record_votes<12>(reads, max_occ, min_votes);
            REQUIRE(res.size() == reads.size());
            for (size_t i = 0; i < reads.size(); ++i)
            {
                REQUIRE(res.status[i] == KMER_B200_QUERY_OK);
                std::map<uint32_t, uint32_t> tally;
                uint32_t hits = 0;
                for (size_t j = 0; j + k <= reads[i].size(); ++j)
                {
                    std::vector<uint32_t> per(texts.size());
                    uint32_t occ = 0;
                    for (size_t t = 0; t < texts.size(); ++t) occ += per[t] = occurrences(texts[t], reads[i], j);
                    if (occ == 0 || (max_occ && occ > max_occ)) continue;
                    ++hits;
                    for (size_t t = 0; t < texts.size(); ++t)
                        if (per[t]) ++tally[uint32_t(t)];
                }
                REQUIRE(res.kmer_hits[i] == hits);
                std::vector<std::pair<uint32_t, uint32_t>> want;
                for (auto [t, v] : tally)
                    if (v >= min_votes) want.emplace_back(t, v);
                std::stable_sort(want.begin(), want.end(), [](auto const& a, auto const& b) { return a.second > b.second; });
                REQUIRE(res[i] == want);
            }
        }

    std::printf("all checks passed\n");
    return 0;
}
