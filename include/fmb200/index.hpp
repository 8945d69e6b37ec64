// fmb200/index.hpp -- host handles with the reference's index / String_c / cursor surface, backed by the device
// image behind the C-ABI (include/fmb200.h).  Header only; calls nothing but the C-ABI.
//
// Mirrors (paths relative to /root/reference/src/fmindex-collection/):
//   fmindex/BiFMIndex.h:17-215        BiFMIndex<Sigma,...>   members bwt, bwtRev, C, size(), locate(), single_locate_step()
//   fmindex/FMIndex.h:14-130          FMIndex<Sigma,...>
//   string/concepts.h:26-87           String_c: size, symbol, rank, prefix_rank, all_ranks, all_ranks_and_prefix_ranks
//   suffixarray/SparseArray.h:44-70   SparseArray built from a range of optional<Entry>
//   fmindex/BiFMIndexCursor.h:13-256  BiFMIndexCursor / LeftBiFMIndexCursor,  fmindex/FMIndexCursor.h:17-60
// Errors: every non-zero C-ABI status becomes std::runtime_error (the reference throws std::runtime_error on
// construction failures, BiFMIndex.h:48-50, utils.h:110,127).  There is no CPU fallback.
#pragma once
#include <filesystem>
#include <algorithm>
#include <array>
#include <cstdint>
#include <memory>
#include <optional>
#include <ranges>
#include <span>
#include <stdexcept>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "../fmb200.h"

namespace fmb200 {

inline void check(int rc) {
    if (rc != FMB_OK) throw std::runtime_error(std::string("fmb200: ") + fmb_last_error() + " (code " + std::to_string(rc) + ")");
}

// ---- concepts.h:12-24 ------------------------------------------------------------------------------------------
template <typename T>
concept Sequence = std::ranges::sized_range<T> && std::ranges::random_access_range<T> && requires(T t) {
    { *t.begin() } -> std::common_with<uint8_t>;
};
template <typename T>
concept Sequences = std::ranges::sized_range<T> && std::ranges::random_access_range<T> && requires(T t) {
    { *t.begin() } -> Sequence;
};

// flattened `Sequences`: the form the C-ABI takes (fmb_queries_upload)
struct FlatSequences {
    std::vector<uint8_t> symbols;
    std::vector<uint64_t> offsets{0};
    size_t size() const { return offsets.size() - 1; }
};
template <Sequences queries_t>
FlatSequences flatten(queries_t const& queries) {
    FlatSequences f;
    size_t total = 0;
    for (auto const& q : queries) total += std::ranges::size(q);
    f.symbols.resize(total);
    f.offsets.reserve(std::ranges::size(queries) + 1);
    size_t at = 0;
    for (auto const& q : queries) {
        for (auto c : q) f.symbols[at++] = static_cast<uint8_t>(c);
        f.offsets.push_back(at);
    }
    return f;
}

// ---- SparseArray (suffixarray/SparseArray.h:44-70) in the generic form the C-ABI takes --------------------------
struct SparseArray {
    using value_t = std::tuple<uint32_t, uint32_t>;
    uint64_t rows{};
    std::vector<uint64_t> bitmap;            // bit i set <=> row i carries a sample
    std::vector<uint32_t> seq, pos;          // samples in row order
    SparseArray() = default;
    template <std::ranges::range range_t>
        requires std::convertible_to<std::ranges::range_value_t<range_t>, std::optional<value_t>>
    explicit SparseArray(range_t const& range) {
        for (auto const& v : range) {
            std::optional<value_t> o = v;
            if (rows % 64 == 0) bitmap.push_back(0);
            if (o) {
                bitmap.back() |= uint64_t{1} << (rows % 64);
                seq.push_back(std::get<0>(*o));
                pos.push_back(std::get<1>(*o));
            }
            ++rows;
        }
    }
};

namespace detail {
struct IndexDeleter {
    void operator()(fmb_index* p) const { fmb_index_destroy(p); }
};
using IndexHandle = std::unique_ptr<fmb_index, IndexDeleter>;
}  // namespace detail

// ---- String_c view of one BWT of a device index (string/concepts.h:26-87) -----------------------------------------
// Every call is one GPU round trip; the batched overloads (spans) are what a caller with many indices should use.
template <size_t TSigma>
struct DeviceString {
    static constexpr size_t Sigma = TSigma;
    fmb_index const* ix{};
    int dir{};
    size_t n{};

    size_t size() const { return n; }
    uint8_t symbol(uint64_t idx) const {
        uint8_t out{};
        check(fmb_string_symbol(ix, dir, &idx, 1, &out));
        return out;
    }
    uint64_t rank(uint64_t idx, uint8_t symb) const {
        uint64_t out{};
        check(fmb_string_rank(ix, dir, &idx, &symb, 1, &out));
        return out;
    }
    uint64_t prefix_rank(uint64_t idx, uint8_t symb) const {
        uint64_t out{};
        check(fmb_string_prefix_rank(ix, dir, &idx, &symb, 1, &out));
        return out;
    }
    auto all_ranks(uint64_t idx) const -> std::array<uint64_t, Sigma> {
        std::array<uint64_t, Sigma> rs{};
        check(fmb_string_all_ranks(ix, dir, &idx, 1, rs.data(), nullptr));
        return rs;
    }
    auto all_ranks_and_prefix_ranks(uint64_t idx) const -> std::tuple<std::array<uint64_t, Sigma>, std::array<uint64_t, Sigma>> {
        std::array<uint64_t, Sigma> rs{}, prs{};
        check(fmb_string_all_ranks(ix, dir, &idx, 1, rs.data(), prs.data()));
        return {rs, prs};
    }
    // batched forms
    void symbol(std::span<uint64_t const> idx, std::span<uint8_t> out) const { check(fmb_string_symbol(ix, dir, idx.data(), idx.size(), out.data())); }
    void rank(std::span<uint64_t const> idx, std::span<uint8_t const> symb, std::span<uint64_t> out) const {
        check(fmb_string_rank(ix, dir, idx.data(), symb.data(), idx.size(), out.data()));
    }
    void prefix_rank(std::span<uint64_t const> idx, std::span<uint8_t const> symb, std::span<uint64_t> out) const {
        check(fmb_string_prefix_rank(ix, dir, idx.data(), symb.data(), idx.size(), out.data()));
    }
    void all_ranks_and_prefix_ranks(std::span<uint64_t const> idx, std::span<uint64_t> rs, std::span<uint64_t> prs) const {
        check(fmb_string_all_ranks(ix, dir, idx.data(), idx.size(), rs.data(), prs.empty() ? nullptr : prs.data()));
    }
};

// index.locate(row) for many rows with one kernel launch (fmb_locate_rows): (seqId, pos, steps) per row
template <typename Rows>
auto locate_rows_raw(fmb_index const* ix, Rows const& rows) -> std::vector<std::tuple<uint32_t, uint32_t, size_t>> {
    size_t const count = std::ranges::size(rows);
    std::vector<uint64_t> r(count), steps(count);
    std::ranges::copy(rows, r.begin());
    std::vector<uint32_t> seq(count), pos(count);
    check(fmb_locate_rows(ix, r.data(), count, seq.data(), pos.data(), steps.data()));
    std::vector<std::tuple<uint32_t, uint32_t, size_t>> out(count);
    for (size_t i = 0; i < count; ++i) out[i] = {seq[i], pos[i], static_cast<size_t>(steps[i])};
    return out;
}
template <typename index_t, typename Rows>
auto locate_rows(index_t const& index, Rows const& rows) { return locate_rows_raw(index.handle(), rows); }

// a range of text: symbols [begin, end) of sequence seq (delimiter excluded), for extract()
struct TextRange {
    uint64_t seq, begin, end;
};
// text extraction (fmb_extract, reconstructText utils.h:672): the symbols of every range, one vector per range
inline auto extract_raw(fmb_index const* ix, std::span<TextRange const> ranges, fmb_stats* stats = nullptr) -> std::vector<std::vector<uint8_t>> {
    size_t const count = ranges.size();
    std::vector<uint64_t> seq(count), begin(count), end(count), offsets(count + 1);
    uint64_t need = 0;
    for (size_t i = 0; i < count; ++i) {
        seq[i] = ranges[i].seq, begin[i] = ranges[i].begin, end[i] = ranges[i].end;
        need += end[i] > begin[i] ? end[i] - begin[i] : 0;
    }
    std::vector<uint8_t> buf(need);
    check(fmb_extract(ix, seq.data(), begin.data(), end.data(), count, buf.data(), need, offsets.data(), stats));
    std::vector<std::vector<uint8_t>> out(count);
    for (size_t i = 0; i < count; ++i) out[i].assign(buf.begin() + offsets[i], buf.begin() + offsets[i + 1]);
    return out;
}

template <typename Index> struct BiFMIndexCursor;
template <typename Index> struct LeftBiFMIndexCursor;
template <typename Index> struct FMIndexCursor;

namespace detail {
// common part of both index kinds
template <size_t TSigma, bool Bidirectional, bool TDelim = true>
struct IndexBase {
    static constexpr size_t Sigma = TSigma;
    static constexpr size_t FirstSymb = TDelim ? 1 : 0;        // BiFMIndex.h:26
    static constexpr bool Delim_v = TDelim;
    using ADEntry = std::tuple<uint32_t, uint32_t>;
    using LEntry = std::tuple<uint32_t, uint32_t, size_t>;

    IndexHandle h;
    DeviceString<Sigma> bwt;
    std::array<size_t, Sigma + 1> C{};

    fmb_index const* handle() const { return h.get(); }
    size_t size() const { return bwt.n; }
    int device() const {
        fmb_index_info info{};
        check(fmb_index_get_info(h.get(), &info));
        return info.device;
    }
    fmb_index_info info() const {
        fmb_index_info i{};
        check(fmb_index_get_info(h.get(), &i));
        return i;
    }

    // BiFMIndex.h:177-202 / FMIndex.h:114-124: (seqId, pos, steps) of one SA row
    auto locate(size_t idx) const -> LEntry {
        auto v = locate_rows(std::array<uint64_t, 1>{idx});
        return v[0];
    }
    // many rows in one launch
    template <typename Rows>
    auto locate_rows(Rows const& rows) const -> std::vector<LEntry> { return fmb200::locate_rows_raw(h.get(), rows); }
    // BiFMIndex.h:204-206
    auto single_locate_step(size_t idx) const -> std::optional<ADEntry> {
        uint64_t row = idx;
        uint8_t has{};
        uint32_t seq{}, pos{};
        check(fmb_sample_value(h.get(), &row, 1, &has, &seq, &pos));
        if (!has) return std::nullopt;
        return ADEntry{seq, pos};
    }

    // symbols per sequence, delimiter excluded (fmb_index_sequence_lengths)
    auto sequence_lengths() const -> std::vector<uint64_t> {
        uint64_t count{};
        check(fmb_index_sequence_count(h.get(), &count));
        std::vector<uint64_t> out(count);
        check(fmb_index_sequence_lengths(h.get(), out.data()));
        return out;
    }
    // symbols [begin, end) of sequence seq, read back from the index on the GPU (fmb_extract)
    auto extract(uint64_t seq, uint64_t begin, uint64_t end) const -> std::vector<uint8_t> {
        TextRange r{seq, begin, end};
        return std::move(extract_raw(h.get(), std::span<TextRange const>(&r, 1))[0]);
    }
    // many ranges in one call
    auto extract(std::span<TextRange const> ranges, fmb_stats* stats = nullptr) const -> std::vector<std::vector<uint8_t>> {
        return extract_raw(h.get(), ranges, stats);
    }

protected:
    void adopt(fmb_index* raw) {
        h.reset(raw);
        fmb_index_info i{};
        check(fmb_index_get_info(raw, &i));
        if (i.sigma != Sigma) throw std::runtime_error("fmb200: index sigma mismatch");
        bwt = DeviceString<Sigma>{raw, 0, static_cast<size_t>(i.n)};
        uint64_t c[Sigma + 1];
        check(fmb_index_get_C(raw, c));
        for (size_t s = 0; s <= Sigma; ++s) C[s] = c[s];
    }
    // text = s0 0 s1 0 ... (utils.h:382-464 createSequences with delimiters)
    template <Sequences seqs_t>
    static std::vector<uint8_t> concat(seqs_t const& input) {
        std::vector<uint8_t> text;
        size_t total = 0;
        for (auto const& s : input) total += std::ranges::size(s) + 1;
        text.reserve(total);
        for (auto const& s : input) {
            for (auto c : s) text.push_back(static_cast<uint8_t>(c));
            text.push_back(0);
        }
        return text;
    }
};
}  // namespace detail

// ---- BiFMIndex (fmindex/BiFMIndex.h:17-215) -----------------------------------------------------------------------
// TDelim = false: BiFMIndex<...>::NoDelim (FirstSymb = 0, omega-sorted text); TReuseRev = true: BiFMIndex<...>::ReuseRev (no bwtRev:
// the BWT of text + reversed text serves both directions).  Both variants are created from BWT bytes (of a reference index, see
// fmb200::attach); the GPU builder behind the Sequences constructor produces delimited indices with a bwtRev.
template <size_t TSigma, bool TDelim = true, bool TReuseRev = false>
struct BiFMIndex : detail::IndexBase<TSigma, true, TDelim> {
    using Base = detail::IndexBase<TSigma, true, TDelim>;
    using Base::Sigma;
    using NoDelim = BiFMIndex<TSigma, false, TReuseRev>;
    using ReuseRev = BiFMIndex<TSigma, TDelim, true>;
    static constexpr bool ReuseRev_v = TReuseRev;
    DeviceString<TSigma> bwtRev;        // ReuseRev: a view of the same BWT (extendRight reads it, BiFMIndexCursor.h fetchRightBwt)

    BiFMIndex() = default;
    BiFMIndex(BiFMIndex&&) noexcept = default;
    auto operator=(BiFMIndex&&) noexcept -> BiFMIndex& = default;

    // BiFMIndex(bwt, bwtRev, SparseArray), BiFMIndex.h:40-51
    BiFMIndex(std::span<uint8_t const> _bwt, std::span<uint8_t const> _bwtRev, SparseArray const& sa, int device = 0)
        requires(!TReuseRev)
    {
        if (_bwt.size() != _bwtRev.size())
            throw std::runtime_error("bwt don't have the same size: " + std::to_string(_bwt.size()) + " " + std::to_string(_bwtRev.size()));
        fmb_index* raw{};
        check(fmb_index_create_ex(&raw, device, Sigma, _bwt.size(), _bwt.data(), _bwtRev.data(), sa.bitmap.data(), sa.seq.data(), sa.pos.data(), sa.seq.size(),
                                  TDelim ? 0u : FMB_INDEX_NO_DELIM));
        init(raw);
    }
    // BiFMIndex(bwt, SparseArray) of the ReuseRev variant, BiFMIndex.h:53-58
    BiFMIndex(std::span<uint8_t const> _bwt, SparseArray const& sa, int device = 0)
        requires(TReuseRev)
    {
        fmb_index* raw{};
        check(fmb_index_create_ex(&raw, device, Sigma, _bwt.size(), _bwt.data(), nullptr, sa.bitmap.data(), sa.seq.data(), sa.pos.data(), sa.seq.size(),
                                  FMB_INDEX_REUSE_REV | (TDelim ? 0u : FMB_INDEX_NO_DELIM)));
        init(raw);
    }
    // BiFMIndex(Sequences, samplingRate, threadNbr), BiFMIndex.h:107-167 (suffix sorting runs on the GPU; threadNbr is
    // accepted for signature compatibility)
    template <Sequences seqs_t>
    BiFMIndex(seqs_t const& input, size_t samplingRate, size_t /*threadNbr*/ = 1, int device = 0)
        requires(TDelim && !TReuseRev)
    {
        auto text = Base::concat(input);
        fmb_index* raw{};
        check(fmb_index_build(&raw, device, Sigma, text.data(), text.size(), static_cast<uint32_t>(samplingRate), 1, 0));
        init(raw);
    }
    // take over an existing handle
    explicit BiFMIndex(fmb_index* raw) { init(raw); }

private:
    void init(fmb_index* raw) {
        Base::adopt(raw);
        fmb_index_info i{};
        check(fmb_index_get_info(raw, &i));
        if (((i.flags & FMB_INDEX_NO_DELIM) != 0) == TDelim || ((i.flags & FMB_INDEX_REUSE_REV) != 0) != TReuseRev)
            throw std::runtime_error("fmb200: index variant (NoDelim / ReuseRev) does not match the index type");
        bwtRev = DeviceString<TSigma>{raw, 1, this->bwt.n};
    }
};

// ---- FMIndex (fmindex/FMIndex.h:14-130) --------------------------------------------------------------------------
template <size_t TSigma>
struct FMIndex : detail::IndexBase<TSigma, false> {
    using Base = detail::IndexBase<TSigma, false>;
    using Base::Sigma;
    FMIndex() = default;
    FMIndex(FMIndex&&) noexcept = default;
    auto operator=(FMIndex&&) noexcept -> FMIndex& = default;
    // FMIndex(bwt, SparseArray), FMIndex.h:28-32
    FMIndex(std::span<uint8_t const> _bwt, SparseArray const& sa, int device = 0) {
        fmb_index* raw{};
        check(fmb_index_create(&raw, device, Sigma, _bwt.size(), _bwt.data(), nullptr, sa.bitmap.data(), sa.seq.data(), sa.pos.data(), sa.seq.size()));
        Base::adopt(raw);
    }
    // FMIndex(Sequences, samplingRate, threadNbr), FMIndex.h:58-112
    template <Sequences seqs_t>
    FMIndex(seqs_t const& input, size_t samplingRate, size_t /*threadNbr*/ = 1, int device = 0) {
        auto text = Base::concat(input);
        fmb_index* raw{};
        check(fmb_index_build(&raw, device, Sigma, text.data(), text.size(), static_cast<uint32_t>(samplingRate), 0, 0));
        Base::adopt(raw);
    }
    explicit FMIndex(fmb_index* raw) { Base::adopt(raw); }
};

// reconstructText (utils.h:672): the delimited text s0 0 s1 0 ... 0 the index was built from (fmb_index_reconstruct_text)
template <typename Index>
auto reconstructText(Index const& index) -> std::vector<uint8_t> {
    std::vector<uint8_t> text(index.size());
    check(fmb_index_reconstruct_text(index.handle(), text.data(), text.size()));
    return text;
}

// ---- persistence (fmindex/diskStorage.h:13-27) -------------------------------------------------------------------------
// saveIndex(index, path) / loadIndex<Index>(path): the flat file of fmb_index_save (BWT bytes + sampled suffix array; the device
// tables are rebuilt when the file is loaded).  Index = fmb200::BiFMIndex<Sigma> or fmb200::FMIndex<Sigma>; a file of the other
// kind or another alphabet size is refused.
template <typename Index>
void saveIndex(Index const& index, std::filesystem::path const& fileName) {
    check(fmb_index_save(index.handle(), fileName.c_str()));
}
template <typename Index>
auto loadIndex(std::filesystem::path const& fileName, int device = 0) -> Index {
    fmb_index* raw{};
    check(fmb_index_load(&raw, device, fileName.c_str()));
    detail::IndexHandle guard{raw};
    fmb_index_info info{};
    check(fmb_index_get_info(raw, &info));
    constexpr bool wantBi = requires(Index const& ix) { ix.bwtRev; };
    if (info.sigma != Index::Sigma || (info.bidirectional != 0) != wantBi) throw std::runtime_error("fmb200::loadIndex: " + fileName.string() + " holds a different index type");
    return Index{guard.release()};
}

// ---- cursors -------------------------------------------------------------------------------------------------------
// BiFMIndexCursor (fmindex/BiFMIndexCursor.h:13-200): value type {index*, lb, lbRev, len, steps}
template <typename Index>
struct BiFMIndexCursor {
    static constexpr size_t Sigma = Index::Sigma;
    static constexpr bool Reversed = false;
    Index const* index{};
    size_t lb{}, lbRev{}, len{}, steps{};
    BiFMIndexCursor() noexcept = default;
    BiFMIndexCursor(Index const& ix) noexcept : BiFMIndexCursor{ix, 0, 0, ix.size(), 0} {}
    BiFMIndexCursor(Index const& ix, size_t lb_, size_t lbRev_, size_t len_, size_t steps_) noexcept
        : index{&ix}, lb{lb_}, lbRev{lbRev_}, len{len_}, steps{steps_} {}
    bool operator==(BiFMIndexCursor const& o) const noexcept { return lb == o.lb && len == o.len; }   // :39-42
    bool empty() const { return len == 0; }
    size_t count() const { return len; }
    auto extendLeft(size_t symb) const -> BiFMIndexCursor { return step(0, symb); }                     // :113-120
    auto extendRight(size_t symb) const -> BiFMIndexCursor { return step(1, symb); }                    // :121-128
    auto extendLeft() const -> std::array<BiFMIndexCursor, Sigma> { return step_all(0); }               // :58-69
    auto extendRight() const -> std::array<BiFMIndexCursor, Sigma> { return step_all(1); }              // :71-82
    size_t symbolLeft() const { return index->bwt.symbol(lb); }                                         // :180-182
    size_t symbolRight() const { return index->bwtRev.symbol(lbRev); }                                  // :183-190

private:
    auto step(int right, size_t symb) const -> BiFMIndexCursor {
        uint64_t cur[4] = {lb, lbRev, len, steps}, out[4];
        uint8_t s = static_cast<uint8_t>(symb);
        check(fmb_cursor_extend(index->handle(), right, cur, &s, 1, out));
        return {*index, out[0], out[1], out[2], out[3]};
    }
    auto step_all(int right) const -> std::array<BiFMIndexCursor, Sigma> {
        uint64_t cur[4] = {lb, lbRev, len, steps};
        std::array<uint64_t, 4 * Sigma> out{};
        check(fmb_cursor_extend_all(index->handle(), right, cur, 1, out.data()));
        std::array<BiFMIndexCursor, Sigma> r;
        for (size_t s = 0; s < Sigma; ++s) r[s] = {*index, out[4 * s], out[4 * s + 1], out[4 * s + 2], out[4 * s + 3]};
        return r;
    }
};

// LeftBiFMIndexCursor (fmindex/BiFMIndexCursor.h:203-256) -- what exact search hands to the delegate
template <typename Index>
struct LeftBiFMIndexCursor {
    static constexpr size_t Sigma = Index::Sigma;
    static constexpr bool Reversed = false;
    Index const* index{};
    size_t lb{}, len{}, steps{};
    LeftBiFMIndexCursor() = default;
    LeftBiFMIndexCursor(BiFMIndexCursor<Index> const& o) : index{o.index}, lb{o.lb}, len{o.len}, steps{o.steps} {}
    LeftBiFMIndexCursor(Index const& ix) : LeftBiFMIndexCursor{ix, 0, ix.size(), 0} {}
    LeftBiFMIndexCursor(Index const& ix, size_t lb_, size_t len_, size_t steps_) : index{&ix}, lb{lb_}, len{len_}, steps{steps_} {}
    bool empty() const { return len == 0; }
    size_t count() const { return len; }
    auto extendLeft(size_t symb) const -> LeftBiFMIndexCursor {                                           // :248-255
        uint64_t at[2] = {lb, lb + len}, r[2];
        uint8_t s[2] = {static_cast<uint8_t>(symb), static_cast<uint8_t>(symb)};
        check(fmb_string_rank(index->handle(), 0, at, s, 2, r));
        return {*index, r[0] + index->C[symb], r[1] - r[0], steps + 1};
    }
};

// FMIndexCursor (fmindex/FMIndexCursor.h:17-60)
template <typename Index>
struct FMIndexCursor {
    static constexpr size_t Sigma = Index::Sigma;
    static constexpr bool Reversed = false;
    Index const* index{};
    size_t lb{}, len{};
    FMIndexCursor() noexcept = default;
    FMIndexCursor(Index const& ix) noexcept : FMIndexCursor{ix, 0, ix.size()} {}
    FMIndexCursor(Index const& ix, size_t lb_, size_t len_) noexcept : index{&ix}, lb{lb_}, len{len_} {}
    bool empty() const { return len == 0; }
    size_t count() const { return len; }
    auto extendLeft(uint8_t symb) const -> FMIndexCursor {                                                // :33-37
        uint64_t at[2] = {lb, lb + len}, r[2];
        uint8_t s[2] = {symb, symb};
        check(fmb_string_rank(index->handle(), 0, at, s, 2, r));
        return {*index, r[0] + index->C[symb], r[1] - r[0]};
    }
};

// search/SelectCursor.h:19-21,48-50,69: which cursor type a search hands to its delegate.  An index type may override
// this by providing member templates/typedefs `cursor_t` / `left_cursor_t` (see fmb200/adapt.hpp).
template <typename Index>
struct select_cursor { using type = BiFMIndexCursor<Index>; using left = LeftBiFMIndexCursor<Index>; };
template <size_t S>
struct select_cursor<FMIndex<S>> { using type = FMIndexCursor<FMIndex<S>>; using left = FMIndexCursor<FMIndex<S>>; };
template <typename Index>
    requires requires { typename Index::cursor_t; typename Index::left_cursor_t; }
struct select_cursor<Index> { using type = typename Index::cursor_t; using left = typename Index::left_cursor_t; };
template <typename Index> using select_cursor_t = typename select_cursor<Index>::type;
template <typename Index> using select_left_cursor_t = typename select_cursor<Index>::left;

}  // namespace fmb200
