// Sequence collections through include/kmer_index.hpp: kmer_index(texts, kmer::collection) over a
// std::vector<std::vector<dna4>> (empty, 1-symbol and short texts included) answers search_batch and search_approx_batch
// with the windows of each text on its own, as a Hamming scan of every text written here; locate() gives (text, offset)
// and a save / load round trip keeps the texts. Exit code 0 = all good. Needs a GPU at run time; compile-only is part of
// the CPU test suite.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <unistd.h>
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

int main()
{
    std::vector<std::vector<alphabet_t>> texts;
    for (size_t len : {5000u, 0u, 1u, 7u, 12000u, 30u, 8000u}) texts.push_back(random_sequence(len));
    std::vector<uint64_t> starts{0};
    std::vector<alphabet_t> concat;
    for (auto const& t : texts)
    {
        concat.insert(concat.end(), t.begin(), t.end());
        starts.push_back(concat.size());
    }
    kmer::kmer_index<alphabet_t, uint32_t, 12> ix(texts, kmer::collection);

    // windows of the texts, windows across two texts (exact and with substitutions) and random reads; lengths 1..100
    std::vector<std::vector<alphabet_t>> queries;
    for (int i = 0; i < 300; ++i)
    {
        size_t m = 1 + next_u32() % 100;
        size_t start = 0;
        if (i % 3 == 0)
            start = next_u32() % (concat.size() - m + 1);
        else if (i % 3 == 1)
        {
            const uint64_t s = starts[1 + next_u32() % (starts.size() - 2)];
            start = size_t(std::min<uint64_t>(s > m / 2 ? s - m / 2 : 0, concat.size() - m));
        }
        else
        {
            queries.push_back(random_sequence(m));
            continue;
        }
        std::vector<alphabet_t> q(concat.begin() + start, concat.begin() + start + m);
        for (int s = 0, d = i % 4; s < d; ++s) q[next_u32() % m].assign_rank(uint8_t(next_u32() % 4));
        queries.push_back(std::move(q));
    }

    auto check = [&](auto const& index, uint32_t e, bool exact) -> int {
        auto batch = exact ? index.search_batch(queries) : index.search_approx_batch(queries, e);
        REQUIRE(batch.size() == queries.size());
        auto where = index.locate(batch);
        REQUIRE(where.size() == batch.positions.size());
        for (size_t i = 0; i < queries.size(); ++i)
        {
            auto const& q = queries[i];
            std::vector<kmer::record_hit> want;
            for (uint32_t r = 0; r < texts.size(); ++r)
                for (size_t p = 0; p + q.size() <= texts[r].size(); ++p)
                {
                    uint32_t d = 0;
                    for (size_t j = 0; j < q.size() && d <= e; ++j) d += texts[r][p + j] != q[j];
                    if (d <= e) want.push_back({r, uint32_t(p)});
                }
            REQUIRE(batch.offsets[i + 1] - batch.offsets[i] == want.size());
            for (size_t j = 0; j < want.size(); ++j)
            {
                const size_t at = batch.offsets[i] + j;
                REQUIRE(where[at] == want[j]);
                REQUIRE(batch.positions[at] == starts[want[j].record] + want[j].offset);
            }
        }
        return 0;
    };
    REQUIRE(check(ix, 0, true) == 0);
    for (uint32_t e : {0u, 2u, 4u}) REQUIRE(check(ix, e, false) == 0);

    const std::string path = "/tmp/kmer_header_collection_" + std::to_string(getpid()) + ".kmerb200";
    ix.save(path);
    auto loaded = kmer::kmer_index<alphabet_t, uint32_t, 12>::load(path);
    std::remove(path.c_str());
    REQUIRE(check(loaded, 2, false) == 0);

    // an index without texts has nothing to locate
    kmer::kmer_index<alphabet_t, uint32_t, 12> plain(concat, 1, KMER_B200_MODE_CORRECT);
    bool threw = false;
    try
    {
        plain.locate(plain.search_batch(queries));
    }
    catch (std::exception const&)
    {
        threw = true;
    }
    REQUIRE(threw);
    std::printf("all checks passed\n");
    return 0;
}
