// Text extraction through the C++ shim: fmb200::reconstructText, BiFMIndex::extract / sequence_lengths and
// PartitionedBiFMIndex::extract across parts, against the sequences the indices were built from.  Needs a GPU; prints "ok".
#include <cstdio>
#include <random>
#include <vector>

#include "fmb200/fmb200.hpp"

static int fails = 0;
#define CHECK(c)                                                        \
    do {                                                                \
        if (!(c)) { std::fprintf(stderr, "FAIL %s:%d %s\n", __FILE__, __LINE__, #c); ++fails; } \
    } while (0)

int main() {
    std::mt19937_64 rng(7);
    std::vector<std::vector<uint8_t>> seqs(300);
    for (auto& s : seqs) {
        s.resize(1 + rng() % 200);
        for (auto& c : s) c = static_cast<uint8_t>(1 + rng() % 4);
    }
    std::vector<uint8_t> text;
    for (auto const& s : seqs) { text.insert(text.end(), s.begin(), s.end()); text.push_back(0); }

    fmb200::BiFMIndex<5> index(seqs, 4);
    CHECK(fmb200::reconstructText(index) == text);
    auto lens = index.sequence_lengths();
    CHECK(lens.size() == seqs.size());
    for (size_t s = 0; s < seqs.size() && s < lens.size(); ++s) CHECK(lens[s] == seqs[s].size());
    CHECK(index.extract(5, 0, seqs[5].size()) == seqs[5]);

    fmb200::FMIndex<5> uni(seqs, 8);
    CHECK(fmb200::reconstructText(uni) == text);

    // two parts (or more): sequence numbers of the whole collection, ranges interleaved across parts
    fmb200::PartitionedBiFMIndex<5> multi(seqs, 4, text.size() / 2 + 1, 1);
    CHECK(multi.parts.size() >= 2);
    std::vector<fmb200::TextRange> ranges;
    for (int k = 0; k < 2000; ++k) {
        uint64_t s = rng() % seqs.size(), len = seqs[s].size();
        uint64_t b = rng() % (len + 1), e = b + rng() % (len - b + 1);
        ranges.push_back({s, b, e});
    }
    ranges.push_back({0, 0, seqs[0].size()});
    ranges.push_back({seqs.size() - 1, 0, seqs.back().size()});
    auto got = multi.extract(ranges);
    CHECK(got.size() == ranges.size());
    for (size_t i = 0; i < ranges.size() && i < got.size(); ++i) {
        auto const& r = ranges[i];
        std::vector<uint8_t> want(seqs[r.seq].begin() + r.begin, seqs[r.seq].begin() + r.end);
        if (got[i] != want) { CHECK(got[i] == want); break; }
    }
    if (fails) return 1;
    std::puts("ok");
    return 0;
}
