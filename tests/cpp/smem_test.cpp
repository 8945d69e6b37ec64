// SMEM search through the C++ shim: the bulk form and the delegate form of fmb200::search_smems report the records of the C-ABI, and
// fmb200::locate_smems the located rows of fmb_locate_smems.  Needs a GPU; prints "ok".
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
    std::mt19937_64 rng(9);
    std::vector<std::vector<uint8_t>> seqs(40);
    for (auto& s : seqs) {
        s.resize(200 + rng() % 800);
        for (auto& c : s) c = static_cast<uint8_t>(1 + rng() % 4);
    }
    fmb200::BiFMIndex<5> index(seqs, 4);
    std::vector<std::vector<uint8_t>> reads(500);
    for (auto& r : reads) {
        auto const& s = seqs[rng() % seqs.size()];
        size_t len = 20 + rng() % 120, p = rng() % (s.size() - 20);
        for (size_t i = 0; i < len; ++i) r.push_back(p + i < s.size() ? s[p + i] : static_cast<uint8_t>(1 + rng() % 4));
        for (int e = 0; e < 3; ++e) r[rng() % r.size()] = static_cast<uint8_t>(1 + rng() % 4);
    }

    // the C-ABI directly
    auto flat = fmb200::flatten(reads);
    fmb_queries* q{};
    fmb200::check(fmb_queries_upload(&q, index.handle(), flat.symbols.data(), flat.offsets.data(), reads.size()));
    fmb_results* r{};
    fmb200::check(fmb_search_smems(index.handle(), q, 0, &r));
    std::vector<fmb_smem> want(fmb_results_count(r));
    fmb200::check(fmb_results_fetch_smems(r, want.data(), want.size()));
    fmb_results* lr{};
    fmb200::check(fmb_locate_smems(index.handle(), r, 3, &lr));
    std::vector<fmb_smem_loc> want_locs(fmb_results_count(lr));
    fmb200::check(fmb_results_fetch_smem_locs(lr, want_locs.data(), want_locs.size()));
    CHECK(!want.empty() && !want_locs.empty());

    auto bulk = fmb200::search_smems(index, reads, 0);
    CHECK(bulk.size() == want.size());
    for (size_t i = 0; i < bulk.size() && i < want.size(); ++i) {
        auto const &a = bulk[i], &b = want[i];
        if (a.qidx != b.qidx || a.begin != b.begin || a.end != b.end || a.lb != b.lb || a.len != b.len) { CHECK(false); break; }
    }
    size_t k = 0;
    fmb200::search_smems(index, reads, 0, [&](size_t qidx, size_t begin, size_t end, auto const& cursor) {
        if (k < want.size()) {
            auto const& b = want[k];
            CHECK(qidx == b.qidx && begin == b.begin && end == b.end && cursor.lb == b.lb && cursor.len == b.len && cursor.steps == end - begin);
        }
        ++k;
    });
    CHECK(k == want.size());
    auto locs = fmb200::locate_smems(index, bulk, 3);
    CHECK(locs.size() == want_locs.size());
    for (size_t i = 0; i < locs.size() && i < want_locs.size(); ++i) {
        auto const &a = locs[i], &b = want_locs[i];
        if (a.qidx != b.qidx || a.begin != b.begin || a.end != b.end || a.seq != b.seq || a.pos != b.pos) { CHECK(false); break; }
    }
    // the longer ones only
    auto longer = fmb200::search_smems(index, reads, 19);
    size_t n19 = 0;
    for (auto const& s : want) n19 += s.end - s.begin >= 19;
    CHECK(longer.size() == n19);
    fmb_results_destroy(lr);
    fmb_results_destroy(r);
    fmb_queries_destroy(q);
    if (fails) return 1;
    std::puts("ok");
    return 0;
}
