// Hit strategies of approximate search through include/kmer_index.hpp: search_approx_batch with approx_hits::all(),
// all_best(), single_best() and strata(s) on a std::vector<std::vector<dna4>> equals a Hamming scan of every window
// written here, distances and best distances included. Exit code 0 = all good. Needs a GPU at run time; compile-only is
// part of the CPU test suite.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <utility>
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

// (position, distance) of every window within e substitutions, ascending
static std::vector<std::pair<uint32_t, uint32_t>> hamming_scan(std::vector<alphabet_t> const& text, std::vector<alphabet_t> const& q,
                                                               uint32_t e)
{
    std::vector<std::pair<uint32_t, uint32_t>> out;
    if (q.empty() || q.size() > text.size()) return out;
    for (size_t p = 0; p + q.size() <= text.size(); ++p)
    {
        uint32_t d = 0;
        for (size_t i = 0; i < q.size(); ++i) d += text[p + i] != q[i];
        if (d <= e) out.emplace_back(uint32_t(p), d);
    }
    return out;
}

// the strategy's hits of one query from the scan; *best = d_min or 0xFF
static std::vector<std::pair<uint32_t, uint32_t>> expected(std::vector<std::pair<uint32_t, uint32_t>> const& all, uint32_t e,
                                                           kmer::approx_hits h, uint32_t* best)
{
    *best = 0xFF;
    if (all.empty()) return {};
    uint32_t dm = 0xFF;
    for (auto const& [p, d] : all) dm = std::min(dm, d);
    *best = dm;
    std::vector<std::pair<uint32_t, uint32_t>> out;
    if (h.strategy == KMER_B200_HITS_SINGLE_BEST)
    {
        for (auto const& hit : all)
            if (hit.second == dm) return {hit};
    }
    const uint32_t lim = h.strategy == KMER_B200_HITS_ALL ? e : h.strategy == KMER_B200_HITS_ALL_BEST ? dm : std::min(e, dm + h.s);
    for (auto const& hit : all)
        if (hit.second <= lim) out.push_back(hit);
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
    auto text = random_sequence(60000);
    for (size_t i = 20000; i < 24000; ++i) text[i].assign_rank(0);  // repeats: several hits at several distances
    kmer::kmer_index<alphabet_t, uint32_t, 12> ix(text, 1, KMER_B200_MODE_CORRECT);

    // text windows with up to 4 substitutions, constant reads and random reads; lengths 1..120
    std::vector<std::vector<alphabet_t>> queries;
    for (int i = 0; i < 240; ++i)
    {
        size_t m = 1 + next_u32() % 120;
        if (i % 5 == 4)
        {
            queries.push_back(random_sequence(m));
            continue;
        }
        if (i % 5 == 3)
        {
            queries.emplace_back(m);
            for (auto& c : queries.back()) c.assign_rank(0);
            queries.back()[next_u32() % m].assign_rank(uint8_t(1 + next_u32() % 3));
            continue;
        }
        size_t start = next_u32() % (text.size() - m + 1);
        std::vector<alphabet_t> q(text.begin() + start, text.begin() + start + m);
        for (int s = 0, d = i % 5; s < d; ++s) q[next_u32() % m].assign_rank(uint8_t(next_u32() % 4));
        queries.push_back(std::move(q));
    }

    const kmer::approx_hits strategies[] = {kmer::approx_hits::all(), kmer::approx_hits::all_best(), kmer::approx_hits::strata(1),
                                            kmer::approx_hits::single_best()};
    for (uint32_t e : {0u, 2u, 4u})
    {
        std::vector<std::vector<std::pair<uint32_t, uint32_t>>> scans;
        for (auto const& q : queries) scans.push_back(hamming_scan(text, q, e));
        for (auto h : strategies)
        {
            auto batch = ix.search_approx_batch(queries, e, h, true);
            REQUIRE(batch.size() == queries.size());
            REQUIRE(batch.distances.size() == batch.positions.size());
            REQUIRE(batch.best_distance.size() == (h.strategy == KMER_B200_HITS_ALL ? 0 : queries.size()));
            for (size_t i = 0; i < queries.size(); ++i)
            {
                uint32_t best = 0;
                auto want = expected(scans[i], e, h, &best);
                REQUIRE(batch.offsets[i + 1] - batch.offsets[i] == want.size());
                for (size_t j = 0; j < want.size(); ++j)
                {
                    REQUIRE(batch.positions[batch.offsets[i] + j] == want[j].first);
                    REQUIRE(batch.distances[batch.offsets[i] + j] == want[j].second);
                }
                if (h.strategy != KMER_B200_HITS_ALL) REQUIRE(batch.best_distance[i] == best);
            }
            auto plain = ix.search_approx_batch(queries, e, h);
            REQUIRE(plain.distances.size() == 0 && plain.positions == batch.positions);
        }
    }
    bool threw = false;
    try
    {
        ix.search_approx_batch(queries, 9, kmer::approx_hits::all_best());
    }
    catch (std::invalid_argument const&)
    {
        threw = true;
    }
    REQUIRE(threw);
    std::printf("all checks passed\n");
    return 0;
}
