// fmb_extract.cu -- text extraction: reconstructText (utils.h:672) and substrings by (sequence, position), on the GPU.
//
// The index holds no copy of the text.  Text is read back with backward LF walks, each starting at an ANCHOR: a text position whose
// BWT row is known.  The anchor table (built on the first call, kept with the index) holds every sampled row with the global position
// start[seq] + pos of its sample, and one anchor per sequence at its delimiter, so every sequence ends in an anchor whatever the
// sampling (text-space, or any row bitmap given to fmb_index_create).  Sorted by position, consecutive anchors cut the text into
// WINDOWS; a window is walked from its upper anchor down to the one below it (or down to the range start), one window per lane.
//
// Sequence layout.  Rows [0, n_delims) are the rows whose suffix starts with a delimiter (C[1] = n_delims): row r is the delimiter
// of some sequence s at position len_s.  Its LF walk runs back through s; it stops at the first sampled row (s, p) -- then
// len_s = p + steps -- or at position 0 of s (BWT symbol 0), where len_s = steps and one more LF step gives the delimiter row of
// sequence s - 1.  A sequence without any sample gets its number from that link; the links are resolved on the host.
#include <algorithm>
#include <cstring>
#include <mutex>
#include <vector>

#include <cub/cub.cuh>

#include "fmb_host.hpp"

namespace fmb {
namespace {

constexpr uint32_t kNone = 0xFFFFFFFFu;

// one thread per delimiter row: walk back to a sampled row or to position 0 of the sequence (see the header comment)
template <class OCC>
__global__ void __launch_bounds__(256) seq_end_kernel(const __grid_constant__ IndexView<OCC> ix, uint32_t nd, uint32_t* __restrict__ seq,
                                                      uint32_t* __restrict__ len, uint32_t* __restrict__ prev) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nd) return;
    row_t row = t;
    uint32_t steps = 0;
    for (;;) {
        const uint4 m = __ldg(ix.marks + (row >> 6));
        const uint64_t bits = (uint64_t)m.x | ((uint64_t)m.y << 32);
        const uint32_t o = row & 63;
        if ((bits >> o) & 1) {
            const uint2 s = __ldg(ix.samples + (m.z + __popcll(bits & low_mask(o))));
            seq[t] = s.x;
            len[t] = s.y + steps;
            prev[t] = kNone;
            return;
        }
        uint32_t c;
        const row_t next = lf_step(ix, ix.occ[0].load(row >> 6, 0), row, c);
        if (c == 0) {                       // position 0 of the sequence: `next` is the delimiter row of the one before
            seq[t] = kNone;
            len[t] = steps;
            prev[t] = next;
            return;
        }
        row = next;
        ++steps;
    }
}

// one thread per 64-row marker word: anchor (start[seq] + pos, row) of every sampled row, at the sample's index
__global__ void __launch_bounds__(256) sample_anchors_kernel(const uint4* __restrict__ marks, const uint2* __restrict__ samples, uint64_t words,
                                                             const uint32_t* __restrict__ start, const uint32_t* __restrict__ len, uint32_t nseq,
                                                             uint32_t* __restrict__ key, uint32_t* __restrict__ val, uint32_t* __restrict__ bad) {
    const uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (w >= words) return;
    const uint4 m = marks[w];
    uint64_t bits = (uint64_t)m.x | ((uint64_t)m.y << 32);
    uint32_t k = m.z;
    while (bits) {
        const uint32_t o = __ffsll((long long)bits) - 1;
        bits &= bits - 1;
        const uint2 s = samples[k];
        if (s.x >= nseq || s.y > len[s.x]) {
            atomicOr(bad, 1u);
            key[k] = 0;
        } else {
            key[k] = start[s.x] + s.y;
        }
        val[k] = (uint32_t)(w * 64 + o);
        ++k;
    }
}

// one thread per range: the anchors covering [gb, ge) are jlo .. jhi with jlo = first anchor > gb, jhi = first anchor >= ge (it exists:
// a range ends at most at its sequence's delimiter, which is an anchor)
__global__ void __launch_bounds__(256) window_count_kernel(const uint32_t* __restrict__ apos, uint32_t na, const uint2* __restrict__ rng,
                                                           uint64_t count, uint32_t* __restrict__ jlo, uint64_t* __restrict__ nwin) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i > count) return;
    if (i == count) { nwin[i] = 0; return; }   // the scan's extra entry: woff[count] = total windows
    const uint2 r = rng[i];
    if (r.y <= r.x) { jlo[i] = 0; nwin[i] = 0; return; }
    uint32_t lo = 0, hi = na;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(apos + mid) <= r.x) lo = mid + 1; else hi = mid; }
    const uint32_t first = lo;
    hi = na;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(apos + mid) < r.y) lo = mid + 1; else hi = mid; }
    jlo[i] = first;
    nwin[i] = (uint64_t)(lo - first) + 1;
}

// K6: window walk.  One window per lane: from the row of anchor j at text position P back down to max(anchor j-1, range start);
// symbols at positions < range end are written to out[off + pos - gb].  Per step, the widest jump that stays inside the window:
// an LF^16 entry of direction 0 (first half of a merged LF^16/LF^32 entry, jstride = 2), an LF^4 entry, else one LF step on the
// occurrence blocks.  A jump entry marked invalid (a delimiter among its symbols) is skipped for the next narrower step.
template <class OCC>
__global__ void __launch_bounds__(256) extract_walk_kernel(const __grid_constant__ IndexView<OCC> ix, const uint2* __restrict__ jump16, uint32_t jstride,
                                                           const uint2* __restrict__ jump4, const uint32_t* __restrict__ apos,
                                                           const uint32_t* __restrict__ arow, const uint2* __restrict__ rng,
                                                           const uint64_t* __restrict__ out_off, const uint32_t* __restrict__ jlo,
                                                           const uint64_t* __restrict__ woff, uint64_t count, uint64_t total,
                                                           uint8_t* __restrict__ out, unsigned long long* __restrict__ counters) {
    const uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    uint32_t requests = 0, steps = 0;
    if (w < total) {
        uint64_t lo = 0, hi = count;                      // largest i with woff[i] <= w (its range has windows)
        while (hi - lo > 1) { const uint64_t mid = (lo + hi) >> 1; if (__ldg(woff + mid) <= w) lo = mid; else hi = mid; }
        const uint64_t i = lo;
        const uint2 r = __ldg(rng + i);
        const uint32_t j = __ldg(jlo + i) + (uint32_t)(w - __ldg(woff + i));
        uint32_t P = __ldg(apos + j);
        row_t row = __ldg(arow + j);
        const uint32_t below = j ? __ldg(apos + j - 1) : 0u;
        const uint32_t stop = max(below, r.x);
        const uint32_t end = min(P, r.y);
        uint8_t* const o = out + (__ldg(out_off + i) - r.x);   // o[pos] for pos in [gb, ge)
        while (P > stop) {
            const uint32_t rem = P - stop;
            if (jump16 && rem >= 16) {
                const uint2 e = __ldg(jump16 + (size_t)row * jstride);
                ++requests;
                if (e.x != kJumpInvalid) {            // 2-bit codes, T[P - 16 + k] in bits 2k (farthest symbol lowest)
                    const uint32_t p0 = P - 16;
#pragma unroll
                    for (uint32_t k = 0; k < 16; ++k)
                        if (p0 + k < end) o[p0 + k] = (uint8_t)(((e.y >> (2 * k)) & 3u) + 1u);
                    row = e.x;
                    P = p0;
                    continue;
                }
            }
            if (jump4 && rem >= 4) {
                const uint2 e = __ldg(jump4 + row);
                ++requests;
                if (e.x != kJumpInvalid) {            // 2-bit codes (DNA layout) or bytes (generic layout), farthest symbol lowest
                    const uint32_t p0 = P - 4;
#pragma unroll
                    for (uint32_t k = 0; k < 4; ++k)
                        if (p0 + k < end)
                            o[p0 + k] = OCC::kSymbolLoad ? (uint8_t)(e.y >> (8 * k)) : (uint8_t)(((e.y >> (2 * k)) & 3u) + 1u);
                    row = e.x;
                    P = p0;
                    continue;
                }
            }
            uint32_t c;
            row = lf_step(ix, ix.occ[0].load(row >> 6, 0), row, c);
            --P;
            if (P < end) o[P] = (uint8_t)c;
            ++steps;
        }
    }
    block_count2(counters, 0, requests, 1, steps);
}

int check_index(const fmb_index* ix) {
    if (!ix) { set_error("NULL index"); return FMB_EINVAL; }
    if (!ix->first_symb) {
        set_error("text extraction needs sequence boundaries; a NoDelim index has none");
        return FMB_EUNSUPPORTED;
    }
    return use_device(ix->device);
}

}  // namespace

// sequence lengths, offsets and delimiter rows (held under ix->anchor_mu, or while the index is being built)
int ensure_layout(const fmb_index* ix) {
    if (ix->layout_ready) return FMB_OK;
    const uint64_t nd = ix->n_delims;
    if (nd == 0) { set_error("index holds no delimiter"); return FMB_EINVAL; }
    if (ix->n_samples == 0) { set_error("index has no sampled suffix array"); return FMB_EINVAL; }
    cudaStream_t st = active_stream(ix);
    DevBuf<uint32_t> d_seq, d_len, d_prev;
    FMB_TRY(d_seq.alloc(nd));
    FMB_TRY(d_len.alloc(nd));
    FMB_TRY(d_prev.alloc(nd));
    if (ix->dna) seq_end_kernel<<<grid_for(nd, 256), 256, 0, st>>>(ix->view_dna(), (uint32_t)nd, d_seq.p, d_len.p, d_prev.p);
    else seq_end_kernel<<<grid_for(nd, 256), 256, 0, st>>>(ix->view_gen(), (uint32_t)nd, d_seq.p, d_len.p, d_prev.p);
    FMB_CUDA(cudaGetLastError());
    note_launches(1);
    std::vector<uint32_t> seq(nd), len(nd), prev(nd);
    FMB_CUDA(cudaMemcpyAsync(seq.data(), d_seq.p, nd * 4, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaMemcpyAsync(len.data(), d_len.p, nd * 4, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaMemcpyAsync(prev.data(), d_prev.p, nd * 4, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    // sequences without a sample: number = number of the sequence before (the delimiter row they link to) + 1, cyclically
    if (nd == 1) seq[0] = 0;
    std::vector<uint32_t> chain;
    for (uint64_t r = 0; r < nd; ++r) {
        uint32_t x = (uint32_t)r;
        chain.clear();
        while (seq[x] == kNone && chain.size() <= nd) {
            chain.push_back(x);
            if (prev[x] >= nd) { set_error("delimiter row %u links to row %u outside the delimiter rows", x, prev[x]); return FMB_EINVAL; }
            x = prev[x];
        }
        if (seq[x] == kNone) { set_error("no sequence of the index holds a sample"); return FMB_EINVAL; }
        for (size_t k = chain.size(); k-- > 0;) seq[chain[k]] = (uint32_t)((seq[prev[chain[k]]] + 1) % nd);
    }
    std::vector<uint64_t> slen(nd, 0), sstart(nd, 0);
    std::vector<uint32_t> srow(nd, kNone);
    for (uint64_t r = 0; r < nd; ++r) {
        if (seq[r] >= nd || srow[seq[r]] != kNone) { set_error("samples name sequence %u twice or out of range", seq[r]); return FMB_EINVAL; }
        srow[seq[r]] = (uint32_t)r;
        slen[seq[r]] = len[r];
    }
    uint64_t pos = 0;
    for (uint64_t s = 0; s < nd; ++s) { sstart[s] = pos; pos += slen[s] + 1; }
    if (pos != ix->n) { set_error("sequence lengths add up to %llu, not n = %llu", (unsigned long long)pos, (unsigned long long)ix->n); return FMB_EINVAL; }
    ix->seq_len = std::move(slen);
    ix->seq_start = std::move(sstart);
    ix->seq_delim_row = std::move(srow);
    ix->layout_ready = true;
    return FMB_OK;
}

namespace {

int ensure_anchors(const fmb_index* ix) {
    FMB_TRY(ensure_layout(ix));
    if (ix->anchor_pos.p) return FMB_OK;
    const uint64_t nd = ix->n_delims, ns = ix->n_samples, na = ns + nd;
    const uint64_t budget = image_budget();
    if (budget && ix->device_bytes() + 8 * na > budget) {
        set_error("anchor table (%llu bytes) does not fit the image budget (%llu of %llu bytes used)", (unsigned long long)(8 * na),
                  (unsigned long long)ix->device_bytes(), (unsigned long long)budget);
        return FMB_ENOMEM;
    }
    cudaStream_t st = active_stream(ix);
    std::vector<uint32_t> h_start(nd), h_len(nd), h_key(nd);
    for (uint64_t s = 0; s < nd; ++s) {
        h_start[s] = (uint32_t)ix->seq_start[s];
        h_len[s] = (uint32_t)ix->seq_len[s];
        h_key[s] = (uint32_t)(ix->seq_start[s] + ix->seq_len[s]);
    }
    DevBuf<uint32_t> d_start, d_len, bad, k0, v0, k1, v1;
    FMB_TRY(d_start.alloc(nd));
    FMB_TRY(d_len.alloc(nd));
    FMB_TRY(bad.alloc(1));
    FMB_TRY(k0.alloc(na));
    FMB_TRY(v0.alloc(na));
    FMB_TRY(k1.alloc(na));
    FMB_TRY(v1.alloc(na));
    FMB_CUDA(cudaMemcpyAsync(d_start.p, h_start.data(), nd * 4, cudaMemcpyHostToDevice, st));
    FMB_CUDA(cudaMemcpyAsync(d_len.p, h_len.data(), nd * 4, cudaMemcpyHostToDevice, st));
    FMB_CUDA(cudaMemcpyAsync(k0.p + ns, h_key.data(), nd * 4, cudaMemcpyHostToDevice, st));
    FMB_CUDA(cudaMemcpyAsync(v0.p + ns, ix->seq_delim_row.data(), nd * 4, cudaMemcpyHostToDevice, st));
    FMB_CUDA(cudaMemsetAsync(bad.p, 0, 4, st));
    const uint64_t words = ix->n / 64 + 1;
    sample_anchors_kernel<<<grid_for(words, 256), 256, 0, st>>>(ix->marks.p, ix->samples.p, words, d_start.p, d_len.p, (uint32_t)nd, k0.p, v0.p, bad.p);
    FMB_CUDA(cudaGetLastError());
    note_launches(1);
    int end_bit = 1;
    while (end_bit < 32 && (uint64_t(1) << end_bit) <= ix->n) ++end_bit;
    cub::DoubleBuffer<uint32_t> keys(k0.p, k1.p), vals(v0.p, v1.p);
    size_t tmp_bytes = 0;
    FMB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys, vals, (int64_t)na, 0, end_bit, st));
    DevBuf<uint8_t> tmp;
    FMB_TRY(tmp.alloc(tmp_bytes));
    FMB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, keys, vals, (int64_t)na, 0, end_bit, st));
    uint32_t h_bad = 0;
    FMB_CUDA(cudaMemcpyAsync(&h_bad, bad.p, 4, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    if (h_bad) { set_error("a sample names a sequence or position outside the collection"); return FMB_EINVAL; }
    ix->anchor_pos = std::move(keys.Current() == k0.p ? k0 : k1);
    ix->anchor_row = std::move(vals.Current() == v0.p ? v0 : v1);
    ix->n_anchors = na;
    return FMB_OK;
}

// Global ranges [gb, ge) (h_rng), range i written at out_off[i] of a device buffer of `bytes` bytes (zeroed first when `zero`), which
// is copied to `out`.
int run_extract(const fmb_index* ix, const std::vector<uint2>& h_rng, const std::vector<uint64_t>& h_off, uint64_t bytes, bool zero,
                uint8_t* out, fmb_stats* stats) {
    cudaStream_t st = active_stream(ix);
    const uint64_t count = h_rng.size();
    fmb_stats s{};
    EventTimer call(st);
    DevBuf<uint2> d_rng;
    DevBuf<uint64_t> d_off, nwin, woff;
    DevBuf<uint32_t> jlo;
    DevBuf<uint8_t> d_out;
    DevBuf<unsigned long long> ctr;
    FMB_TRY(d_rng.alloc(count));
    FMB_TRY(d_off.alloc(count));
    FMB_TRY(jlo.alloc(count));
    FMB_TRY(nwin.alloc(count + 1));
    FMB_TRY(woff.alloc(count + 1));
    FMB_TRY(d_out.alloc(bytes));
    FMB_TRY(ctr.alloc(2));
    FMB_CUDA(cudaMemcpyAsync(d_rng.p, h_rng.data(), count * sizeof(uint2), cudaMemcpyHostToDevice, st));
    FMB_CUDA(cudaMemcpyAsync(d_off.p, h_off.data(), count * 8, cudaMemcpyHostToDevice, st));
    FMB_CUDA(cudaMemsetAsync(ctr.p, 0, 2 * sizeof(unsigned long long), st));
    if (zero) FMB_CUDA(cudaMemsetAsync(d_out.p, 0, bytes, st));
    s.h2d_bytes = count * (sizeof(uint2) + 8);
    window_count_kernel<<<grid_for(count + 1, 256), 256, 0, st>>>(ix->anchor_pos.p, (uint32_t)ix->n_anchors, d_rng.p, count, jlo.p, nwin.p);
    FMB_CUDA(cudaGetLastError());
    size_t tmp_bytes = 0;
    FMB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, nwin.p, woff.p, (int64_t)(count + 1), st));
    DevBuf<uint8_t> tmp;
    FMB_TRY(tmp.alloc(tmp_bytes));
    FMB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, nwin.p, woff.p, (int64_t)(count + 1), st));
    uint64_t total = 0;
    FMB_CUDA(cudaMemcpyAsync(&total, woff.p + count, 8, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    note_launches(2);
    if (total) {
        // LF^16 entries of direction 0 (DNA layout; the first half of merged LF^16/LF^32 entries) and LF^4 entries
        const uint2* j16 = ix->dna ? ix->jump[0].p : nullptr;
        const uint32_t jstride = ix->jump_shift[0] ? 2u : 1u;
        const uint2* j4 = ix->jump4[0].p;
        EventTimer walk(st);
        if (ix->dna)
            extract_walk_kernel<<<grid_for(total, 256), 256, 0, st>>>(ix->view_dna(), j16, jstride, j4, ix->anchor_pos.p, ix->anchor_row.p, d_rng.p,
                                                                      d_off.p, jlo.p, woff.p, count, total, d_out.p, ctr.p);
        else
            extract_walk_kernel<<<grid_for(total, 256), 256, 0, st>>>(ix->view_gen(), j16, jstride, j4, ix->anchor_pos.p, ix->anchor_row.p, d_rng.p,
                                                                      d_off.p, jlo.p, woff.p, count, total, d_out.p, ctr.p);
        FMB_CUDA(cudaGetLastError());
        note_launches(1);
        s.main_kernel_ms = walk.stop();
    }
    unsigned long long h_ctr[2] = {0, 0};
    FMB_CUDA(cudaMemcpyAsync(h_ctr, ctr.p, sizeof h_ctr, cudaMemcpyDeviceToHost, st));
    if (bytes) FMB_CUDA(cudaMemcpyAsync(out, d_out.p, bytes, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    s.kernel_ms = call.stop();
    s.line_requests = h_ctr[0];
    s.lf_steps = h_ctr[1];
    s.d2h_bytes = bytes;
    if (stats) *stats = s;
    return FMB_OK;
}

}  // namespace
}  // namespace fmb

using namespace fmb;

extern "C" {

int fmb_index_sequence_count(const fmb_index* ix, uint64_t* count) {
    if (!count) { set_error("NULL argument"); return FMB_EINVAL; }
    FMB_TRY(check_index(ix));
    *count = ix->n_delims;
    return FMB_OK;
}

int fmb_index_sequence_lengths(const fmb_index* ix, uint64_t* lengths) {
    if (!lengths) { set_error("NULL argument"); return FMB_EINVAL; }
    FMB_TRY(check_index(ix));
    std::lock_guard<std::mutex> lk(ix->anchor_mu);
    FMB_TRY(ensure_layout(ix));
    std::copy(ix->seq_len.begin(), ix->seq_len.end(), lengths);
    return FMB_OK;
}

int fmb_extract(const fmb_index* ix, const uint64_t* seq, const uint64_t* begin, const uint64_t* end, uint64_t count,
                uint8_t* out, uint64_t capacity, uint64_t* offsets, fmb_stats* stats) {
    if (!offsets || (count && (!seq || !begin || !end))) { set_error("NULL argument"); return FMB_EINVAL; }
    FMB_TRY(check_index(ix));
    if (stats) *stats = fmb_stats{};
    {
        std::lock_guard<std::mutex> lk(ix->anchor_mu);
        FMB_TRY(ensure_anchors(ix));
    }
    std::vector<uint2> rng(count);
    std::vector<uint64_t> off(count);
    uint64_t total = 0;
    offsets[count] = 0;
    for (uint64_t i = 0; i < count; ++i) {
        if (seq[i] >= ix->n_delims) {
            set_error("seq[%llu] = %llu: the index holds %llu sequences", (unsigned long long)i, (unsigned long long)seq[i], (unsigned long long)ix->n_delims);
            return FMB_EINVAL;
        }
        const uint64_t len = ix->seq_len[seq[i]];
        if (begin[i] > end[i] || end[i] > len) {
            set_error("range %llu = [%llu, %llu) of sequence %llu (length %llu) is invalid", (unsigned long long)i, (unsigned long long)begin[i],
                      (unsigned long long)end[i], (unsigned long long)seq[i], (unsigned long long)len);
            return FMB_EINVAL;
        }
        const uint64_t st = ix->seq_start[seq[i]];
        rng[i] = make_uint2((uint32_t)(st + begin[i]), (uint32_t)(st + end[i]));
        off[i] = offsets[i] = total;
        total += end[i] - begin[i];
    }
    offsets[count] = total;
    if (capacity < total) {
        set_error("output capacity %llu < %llu bytes needed", (unsigned long long)capacity, (unsigned long long)total);
        return FMB_EINVAL;
    }
    if (total && !out) { set_error("NULL argument"); return FMB_EINVAL; }
    if (count == 0) return FMB_OK;
    return run_extract(ix, rng, off, total, false, out, stats);
}

int fmb_index_reconstruct_text(const fmb_index* ix, uint8_t* out, uint64_t capacity) {
    FMB_TRY(check_index(ix));
    if (!out) { set_error("NULL argument"); return FMB_EINVAL; }
    if (capacity < ix->n) {
        set_error("output capacity %llu < n = %llu", (unsigned long long)capacity, (unsigned long long)ix->n);
        return FMB_EINVAL;
    }
    {
        std::lock_guard<std::mutex> lk(ix->anchor_mu);
        FMB_TRY(ensure_anchors(ix));
    }
    // one range per sequence at its own offset; the delimiters are the zeros the output buffer starts with
    const uint64_t nd = ix->n_delims;
    std::vector<uint2> rng(nd);
    std::vector<uint64_t> off(nd);
    for (uint64_t s = 0; s < nd; ++s) {
        off[s] = ix->seq_start[s];
        rng[s] = make_uint2((uint32_t)off[s], (uint32_t)(off[s] + ix->seq_len[s]));
    }
    return run_extract(ix, rng, off, ix->n, true, out, nullptr);
}

}  // extern "C"
