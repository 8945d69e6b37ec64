// fmb200/smem.hpp -- super-maximal exact matches (SMEMs) of a query batch, on the GPU (fmb_search_smems / fmb_locate_smems).
//
// [begin, end) of a query Q occurs when Q[begin:end] holds no symbol 0 or >= Sigma and is a substring of one sequence of the
// collection; it is an SMEM when it occurs and can be made longer on neither side and still occur (begin == 0 / end == |Q| count as
// blocked).  lb / len is the SA interval of Q[begin:end] in the forward BWT, the interval exact search reports for it.  The reference
// library has no counterpart: these are the seeds a BWA-MEM-style mapper places reads with when they differ too much for k-error search.
#pragma once
#include <memory>

#include "search.hpp"

namespace fmb200 {

// The records of search_smems (ordered by qidx, then begin), together with the device result set locate_smems reads.
struct SmemRecords : std::vector<fmb_smem> {
    std::shared_ptr<fmb_results> device;
};

// every SMEM of every query with end - begin >= min_len
template <typename index_t, Sequences queries_t>
SmemRecords search_smems(index_t const& index, queries_t const& queries, size_t min_len = 1, fmb_stats* stats = nullptr) {
    auto flat = flatten(queries);
    auto q = detail::upload(index.handle(), flat);
    fmb_results* r{};
    check(fmb_search_smems(index.handle(), q.get(), static_cast<uint32_t>(std::min<size_t>(min_len, UINT32_MAX)), &r));
    SmemRecords out;
    out.device = std::shared_ptr<fmb_results>(r, fmb_results_destroy);
    if (stats) check(fmb_results_get_stats(r, stats));
    out.resize(fmb_results_count(r));
    check(fmb_results_fetch_smems(r, out.data(), out.size()));
    return out;
}

// delegate(qidx, begin, end, cursor) per SMEM in record order; the cursor is left-only: no lbRev is reported
template <typename index_t, Sequences queries_t, typename delegate_t>
void search_smems(index_t const& index, queries_t const& queries, size_t min_len, delegate_t&& delegate) {
    for (auto const& s : search_smems(index, queries, min_len)) {
        fmb_hit h{s.qidx, s.lb, 0, s.len, s.end - s.begin, 0};
        delegate(static_cast<size_t>(s.qidx), static_cast<size_t>(s.begin), static_cast<size_t>(s.end), detail::make_left_cursor(index, h));
    }
}

// per SMEM the first min(len, max_occ) rows of its interval, located: (qidx, begin, end, seq, pos) with pos = position of Q[begin]
template <typename index_t>
std::vector<fmb_smem_loc> locate_smems(index_t const& index, SmemRecords const& smems, uint64_t max_occ = UINT64_MAX) {
    fmb_results* r{};
    check(fmb_locate_smems(index.handle(), smems.device.get(), max_occ, &r));
    detail::ResultsHandle res{r};
    std::vector<fmb_smem_loc> out(fmb_results_count(r));
    check(fmb_results_fetch_smem_locs(r, out.data(), out.size()));
    return out;
}

}  // namespace fmb200
