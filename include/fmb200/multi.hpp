// fmb200/multi.hpp -- one index replica per GPU (built once, copied over peer memory), queries sharded contiguously.
// SURVEY.md §8(e): queries are independent, the index is replicated, there is NO collective on the search path;
// every GPU is driven by its own host thread.
#pragma once
#include <exception>
#include <thread>

#include "search.hpp"

namespace fmb200 {

// contiguous shard [begin, end) of `count` items for `rank` of `world` (sizes differ by at most one)
inline std::pair<size_t, size_t> shard_range(size_t count, size_t rank, size_t world) {
    size_t const base = count / world, rest = count % world;
    size_t const begin = rank * base + std::min(rank, rest);
    return {begin, begin + base + (rank < rest ? 1 : 0)};
}

template <size_t Sigma>
struct ReplicatedBiFMIndex {
    std::vector<BiFMIndex<Sigma>> replicas;     // replicas[g] lives on device g

    // the image is built ONCE (on device 0) and copied to the other devices over peer memory (fmb_index_replicate)
    ReplicatedBiFMIndex(std::span<uint8_t const> bwt, std::span<uint8_t const> bwtRev, SparseArray const& sa, int n_devices = fmb_device_count()) {
        if (n_devices < 1) throw std::runtime_error("fmb200: no CUDA device (libfmb200 has no CPU fallback)");
        replicas.emplace_back(bwt, bwtRev, sa, 0);
        replicate(n_devices);
    }
    // replicas of an index that exists already (it becomes replica 0)
    explicit ReplicatedBiFMIndex(BiFMIndex<Sigma>&& first, int n_devices = fmb_device_count()) {
        replicas.push_back(std::move(first));
        replicate(n_devices);
    }
    size_t world() const { return replicas.size(); }

    // One call for the whole batch (fmb_search_and_locate_multi): the queries are split into contiguous shards of ceil(Q / G), every
    // replica searches + locates its shard at the same time, the located rows (qidx, seq, pos + offset, e; qidx = index in the whole
    // batch) come back shard after shard, i.e. grouped by ascending ranges of qidx.  scheme == nullptr selects exact search.
    template <Sequences queries_t, detail::SchemeLike scheme_t = search_scheme::Scheme>
    std::vector<fmb_loc32> search_and_locate(queries_t const& queries, bool edit = false, scheme_t const* scheme = nullptr,
                                             std::vector<size_t> const* partition = nullptr, fmb_stats* stats = nullptr) const {
        auto flat = flatten(queries);
        detail::FlatScheme fs;
        if (scheme) fs = detail::flatten(*scheme, *partition);
        size_t const G = world();
        std::vector<fmb_index const*> handles;
        for (auto const& r : replicas) handles.push_back(r.handle());
        size_t cap = std::max<size_t>((flat.size() + G - 1) / G * 2, 1024);
        std::vector<uint64_t> n_out(G);
        for (;;) {
            std::vector<fmb_loc32> out(cap * G);
            int rc = fmb_search_and_locate_multi(handles.data(), static_cast<uint32_t>(G), flat.symbols.data(), flat.offsets.data(), flat.size(), edit ? 1 : 0,
                                                 fs.n_searches, fs.n_parts, fs.pi.data(), fs.l.data(), fs.u.data(), fs.partition.data(), out.data(), cap,
                                                 n_out.data(), stats);
            if (rc == FMB_EOVERFLOW) {
                size_t const need = *std::max_element(n_out.begin(), n_out.end());
                if (need > cap) { cap = need; continue; }
            }
            check(rc);
            std::vector<fmb_loc32> all;
            for (size_t g = 0; g < G; ++g) all.insert(all.end(), out.begin() + g * cap, out.begin() + g * cap + n_out[g]);
            return all;
        }
    }

    // runs `fn(replica, shard_of_queries, first_qidx) -> std::vector<fmb_hit>` on every GPU and concatenates
    template <typename queries_t, typename Fn>
    std::vector<fmb_hit> run_sharded(queries_t const& queries, Fn&& fn) const {
        size_t const G = world(), Q = std::ranges::size(queries);
        std::vector<std::vector<fmb_hit>> parts(G);
        std::vector<std::exception_ptr> errs(G);
        std::vector<std::thread> threads;
        for (size_t g = 0; g < G; ++g) {
            threads.emplace_back([&, g] {
                try {
                    auto [b, e] = shard_range(Q, g, G);
                    auto shard = std::ranges::subrange(std::ranges::begin(queries) + b, std::ranges::begin(queries) + e);
                    parts[g] = fn(replicas[g], shard);
                    for (auto& h : parts[g]) h.qidx += b;
                } catch (...) { errs[g] = std::current_exception(); }
            });
        }
        for (auto& t : threads) t.join();
        for (auto& e : errs)
            if (e) std::rethrow_exception(e);
        std::vector<fmb_hit> all;
        for (auto& p : parts) all.insert(all.end(), p.begin(), p.end());
        return all;
    }

private:
    void replicate(int n_devices) {
        for (int g = 1; g < n_devices; ++g) {
            fmb_index* raw{};
            check(fmb_index_replicate(replicas[0].handle(), g, &raw));
            replicas.emplace_back(raw);
        }
    }

public:
    template <Sequences queries_t>
    std::vector<fmb_hit> search_exact(queries_t const& queries) const {
        return run_sharded(queries, [](auto const& ix, auto const& shard) { return search_no_errors::search_bulk(ix, shard); });
    }
    template <bool Edit, Sequences queries_t>
    std::vector<fmb_hit> search_scheme(queries_t const& queries, search_scheme::Scheme const& scheme, std::vector<size_t> const& partition) const {
        return run_sharded(queries, [&](auto const& ix, auto const& shard) { return search_ng26::search_bulk<Edit>(ix, shard, scheme, partition); });
    }
};

// A collection too large for one index (n >= 2^32 - 64 rows: the reference switches to 64-bit suffix arrays, utils.h:243-247; the
// device image keeps 32-bit rows): the sequences are split, in order, into parts of at most `max_part_symbols` symbols (delimiters
// included), one BiFMIndex per part, parts placed round-robin on `n_devices` devices (several parts on one device need an image budget
// that lets them fit: fmb_set_image_budget).  search_and_locate searches the whole batch in every part (fmb_search_and_locate_parts)
// and returns the located rows with the sequence numbers of the whole collection -- the rows one index over everything would return,
// as a multiset, grouped by part.
template <size_t Sigma>
struct PartitionedBiFMIndex {
    std::vector<BiFMIndex<Sigma>> parts;
    std::vector<uint64_t> seq_base;             // number of the first sequence of every part

    static constexpr uint64_t kMaxPartSymbols = 0xFFFFFFFFull - 64;

    template <Sequences sequences_t>
    PartitionedBiFMIndex(sequences_t const& sequences, size_t samplingRate, uint64_t max_part_symbols = kMaxPartSymbols - 1,
                         int n_devices = fmb_device_count()) {
        if (n_devices < 1) throw std::runtime_error("fmb200: no CUDA device (libfmb200 has no CPU fallback)");
        if (max_part_symbols >= kMaxPartSymbols) max_part_symbols = kMaxPartSymbols - 1;
        auto first = std::ranges::begin(sequences);
        auto const end = std::ranges::end(sequences);
        uint64_t seq_no = 0;
        while (first != end) {
            auto last = first;
            uint64_t symbols = 0, count = 0;
            while (last != end && (count == 0 || symbols + std::ranges::size(*last) + 1 <= max_part_symbols)) {
                symbols += std::ranges::size(*last) + 1;
                ++last;
                ++count;
            }
            if (symbols > kMaxPartSymbols - 1) throw std::runtime_error("fmb200: one sequence alone exceeds 2^32 - 64 symbols");
            std::vector<std::vector<uint8_t>> group;
            for (auto it = first; it != last; ++it) group.emplace_back(std::ranges::begin(*it), std::ranges::end(*it));
            seq_base.push_back(seq_no);
            parts.emplace_back(group, samplingRate, 1, static_cast<int>(parts.size() % static_cast<size_t>(n_devices)));
            seq_no += count;
            first = last;
        }
    }
    size_t size() const {
        size_t n = 0;
        for (auto const& p : parts) n += p.size();
        return n;
    }

    // text extraction with sequence numbers of the whole collection: every range goes to the part that holds its sequence
    auto extract(std::span<TextRange const> ranges, fmb_stats* stats = nullptr) const -> std::vector<std::vector<uint8_t>> {
        std::vector<std::vector<TextRange>> local(parts.size());
        std::vector<std::vector<size_t>> where(parts.size());
        for (size_t i = 0; i < ranges.size(); ++i) {
            size_t const p = static_cast<size_t>(std::upper_bound(seq_base.begin(), seq_base.end(), ranges[i].seq) - seq_base.begin()) - 1;
            local[p].push_back({ranges[i].seq - seq_base[p], ranges[i].begin, ranges[i].end});
            where[p].push_back(i);
        }
        std::vector<std::vector<uint8_t>> out(ranges.size());
        if (stats) *stats = fmb_stats{};
        for (size_t p = 0; p < parts.size(); ++p) {
            if (local[p].empty()) continue;
            fmb_stats s{};
            auto got = parts[p].extract(std::span<TextRange const>(local[p]), &s);
            for (size_t k = 0; k < got.size(); ++k) out[where[p][k]] = std::move(got[k]);
            if (stats) stats->line_requests += s.line_requests, stats->lf_steps += s.lf_steps, stats->kernel_ms += s.kernel_ms;
        }
        return out;
    }

    template <Sequences queries_t, detail::SchemeLike scheme_t = search_scheme::Scheme>
    std::vector<fmb_loc32> search_and_locate(queries_t const& queries, bool edit = false, scheme_t const* scheme = nullptr,
                                             std::vector<size_t> const* partition = nullptr, fmb_stats* stats = nullptr) const {
        auto flat = flatten(queries);
        detail::FlatScheme fs;
        if (scheme) fs = detail::flatten(*scheme, *partition);
        size_t const P = parts.size();
        std::vector<fmb_index const*> handles;
        for (auto const& p : parts) handles.push_back(p.handle());
        size_t cap = std::max<size_t>(flat.size() * 2, 1024);
        std::vector<uint64_t> n_out(P);
        for (;;) {
            std::vector<fmb_loc32> out(cap * P);
            int rc = fmb_search_and_locate_parts(handles.data(), static_cast<uint32_t>(P), seq_base.data(), flat.symbols.data(), flat.offsets.data(), flat.size(),
                                                 edit ? 1 : 0, fs.n_searches, fs.n_parts, fs.pi.data(), fs.l.data(), fs.u.data(), fs.partition.data(), out.data(), cap,
                                                 n_out.data(), stats);
            if (rc == FMB_EOVERFLOW) {
                size_t const need = *std::max_element(n_out.begin(), n_out.end());
                if (need > cap) { cap = need; continue; }
            }
            check(rc);
            std::vector<fmb_loc32> all;
            for (size_t g = 0; g < P; ++g) all.insert(all.end(), out.begin() + g * cap, out.begin() + g * cap + n_out[g]);
            return all;
        }
    }
};

}  // namespace fmb200
