// fmb_smem.cu -- K7: super-maximal exact matches (SMEMs) of a query batch, their located rows, and their C-ABI (include/fmb200.h).
//
// Definition.  [i, j) of a query Q of length m occurs when Q[i:j] holds no non-matching symbol (0 or >= sigma) and is a substring of
// one sequence of the collection; it is an SMEM when it occurs and neither [i-1, j) nor [i, j+1) does (i == 0 and j == m count as
// blocked).  SMEMs are the occurring intervals that are maximal under containment: their starts and ends both increase strictly.
//
// Algorithm (per query, linear in its length): a right phase extends Q[x:j] to the right until it stops occurring -- [x, j) is then an
// SMEM -- and a left phase finds the smallest b with Q[b:j+1] occurring, starting from Q[j] alone and extending left no further than
// x + 1 (extending by Q[x] is known to fail).  The next right phase continues from the cursor of Q[b:j+1], which is why both phases
// use the bidirectional step extend_bi and the left phase keeps lb_rev.  A right phase that starts from the whole index takes its
// first bikmer_k symbols in one lookup of the bidirectional k-mer table where the image has one (a missing k-mer takes single steps).
//
// Work distribution.  The work per read is very uneven: an exact read has one SMEM and costs about m steps, a read of unrelated
// sequence has about m - log_4(n) overlapping SMEMs of about log_4(n) symbols and costs about ten times that.  So the kernel is a
// persistent grid of lanes, one query per lane, and a lane that finishes a query takes the next one from a global counter (one atomic
// per group of lanes that finish together).  All lanes run the same loop body: a resolve step that settles everything not needing the
// index (phase changes, reports, text-path comparisons, taking a new query), then ONE extend_bi step for every lane that wants one,
// so lanes in different phases of different queries still issue their occurrence-table lookups together.  Records are appended to a
// staging list in the order they are found, with the number of the record within its query; a per-query count, its prefix sum and
// one scatter put them in (qidx, begin) order.  The staging list grows and the search reruns when it was too small.
//
// Text path (FMB_TEXT_CHECK: DNA layout with delimiter; queries without a non-matching symbol).  Once the interval of Q[x:j] is one
// row, Q[x:j] occurs once, at the text position g of that row (row_pos: suffix array or locate shortcut), and Q[x:j+1] occurs iff
// the text continues with Q[j] inside the same sequence: the rest of the right phase compares the 2-bit text with the packed query
// 16 symbols (one 32-bit word) at a time, the first mismatch coming from the XOR of the two words; the row does not change.  The
// text gives delimiter positions the code of symbol 1, so every comparison is bounded by the sequence borders, never by codes.
// Only right phases that start from the whole index take the text path (the first SMEM of a read, and the first after a non-matching
// symbol): that phase covers the whole of an exact read and the stretch up to the first edit of the others.  Left phases, and the
// right phases that continue from them, stay on the index.  There the interval becomes one row only a few symbols before the phase
// ends, so the chain of dependent lookups that finds the row's text position (locate shortcut, sample, sequence start) costs more than
// the steps it replaces -- and while one lane waits on that chain, the other lanes of its warp wait with it (measured: DESIGN §3 K7).
#include <cooperative_groups.h>

#include <algorithm>
#include <cstring>
#include <vector>

#include "fmb_host.hpp"

namespace cg = cooperative_groups;

namespace fmb {
namespace {

constexpr uint32_t kNone = 0xFFFFFFFFu;

struct SmemStage {                // one record as found: query, its number within the query, the SMEM and (seq, pos) of the text path
    uint32_t q, k, begin, end, lb, len, seq, pos;
};

struct SmemArgs {
    const uint8_t* qsym;
    const uint64_t* qoff;
    const uint8_t* qflags;        // DNA layout: 1 = the query holds a non-matching symbol
    const uint32_t* qpk;          // DNA layout: 2-bit packed queries
    uint32_t nq, min_len;
    const uint4* bikmer;          // nullptr: no k-mer seeding
    uint32_t bikmer_k, bikmer_base;   // base 0: 2-bit key (DNA layout)
    const uint32_t* text32;       // nullptr: no text path
    RowPosView rowpos;
    SmemStage* stage;
    unsigned long long cap;       // records the staging list holds
    uint32_t* counts;             // per query: SMEMs reported
    unsigned long long* ctr;      // [0] extensions [1] occ lookups [2] line requests [3] records found [4] next query
};

enum : uint32_t { PH_NEW, PH_RIGHT, PH_STOP, PH_LEFT0, PH_LEFT, PH_IDLE, PH_DONE };   // PH_DONE: no query left

__device__ __forceinline__ uint32_t sym_mask(uint32_t cnt) { return cnt >= 16 ? 0xFFFFFFFFu : (1u << (2 * cnt)) - 1u; }
// 16 symbols of a 2-bit stream from symbol position p on (the stream is padded: the word after the last one exists)
__device__ __forceinline__ uint32_t word_at(const uint32_t* s, uint64_t p) {
    const uint64_t w = p >> 4;
    return __funnelshift_r(__ldg(s + w), __ldg(s + w + 1), 2 * (uint32_t)(p & 15));
}

template <class OCC>
__global__ void __launch_bounds__(256) smem_kernel(const __grid_constant__ IndexView<OCC> ix, const __grid_constant__ SmemArgs a) {
    uint32_t ext = 0, look = 0, lines = 0;
    uint32_t q = 0, m = 0, x = 0, j = 0, b = 0, k = 0, ph = PH_IDLE;
    uint64_t off = 0;
    bool text = false;            // this query may take the text path
    bool fresh = false;           // the right phase started from the whole index (not from a left phase)
    Cursor cur{0, 0, 0, 0};
    uint32_t tg = kNone, tbeg = 0, tend = 0, tseq = 0;     // text mode: Q[x] lies at tg, in sequence tseq = text [tbeg, tend)
    const Cursor whole{0, 0, ix.n, 0};
    auto sym = [&](uint32_t p) -> uint32_t { return __ldg(a.qsym + off + p); };
    auto matches = [&](uint32_t c) { return c >= 1 && c < ix.sigma; };
    // text position of the suffix of `row` and the borders of its sequence
    auto text_pos = [&](row_t row) -> uint32_t {
        const RowPos p = row_pos<true>(a.rowpos, row, lines);
        tseq = p.seq;
        tbeg = p.start;
        tend = __ldg(a.rowpos.seq_start + tseq + 1) - 1;          // the sequence's delimiter
        lines += 1;
        return p.g;
    };
    for (;;) {
        // ---- resolve: everything up to the next extension this lane needs --------------------------------------------------------
        bool want = false;
        uint32_t wsym = 0;
        int wright = 0;
        Cursor base = whole;
        while (!want && ph != PH_DONE) {
            if (ph == PH_IDLE) {
                cg::coalesced_group g = cg::coalesced_threads();
                unsigned long long t = 0;
                if (g.thread_rank() == 0) t = atomicAdd(a.ctr + 4, (unsigned long long)g.size());
                t = g.shfl(t, 0) + g.thread_rank();
                if (t >= a.nq) { ph = PH_DONE; break; }
                q = (uint32_t)t;
                off = a.qoff[q];
                m = (uint32_t)(a.qoff[q + 1] - off);
                x = 0; k = 0; tg = kNone;
                text = !OCC::kSymbolLoad && a.text32 && !a.qflags[q];      // the text tables exist on the DNA layout only
                ph = PH_NEW;
            } else if (ph == PH_NEW) {
                if (x >= m) { a.counts[q] = k; ph = PH_IDLE; continue; }
                const uint32_t c = sym(x);
                if (!matches(c)) { ++x; continue; }
                if (a.bikmer && x + a.bikmer_k <= m) {
                    uint32_t key = 0, mul = 1;
                    bool ok = true;
                    for (uint32_t p = 0; p < a.bikmer_k && ok; ++p) {
                        const uint32_t s = sym(x + p);
                        ok = matches(s);
                        key += a.bikmer_base ? (s - 1) * mul : (s - 1) << (2 * p);
                        mul *= a.bikmer_base;
                    }
                    if (ok) {
                        const uint4 e = __ldg(a.bikmer + key);
                        lines += 1;
                        ext += e.w >> 16;
                        look += e.w & 0xFFFFu;
                        if (e.z) {
                            cur = Cursor{e.x, e.y, e.z, a.bikmer_k};
                            j = x + a.bikmer_k;
                            ph = PH_RIGHT;
                            fresh = true;
                            continue;
                        }
                    }
                }
                want = true; wsym = c; wright = 1; base = whole;
            } else if (ph == PH_RIGHT) {
                if (text && fresh && cur.len == 1 && j < m) {
                    // Q[x:j] occurs once, at tg: the text decides how far it extends
                    tg = text_pos(cur.lb);
                    uint32_t t = tg + (j - x);
                    uint32_t lim = min(m - j, tend - t);
                    while (lim) {
                        const uint32_t cnt = min(16u, lim);
                        const uint32_t d = (word_at(a.qpk, off + j) ^ word_at(a.text32, t)) & sym_mask(cnt);
                        lines += 1;
                        if (d) { j += (uint32_t)(__ffs(d) - 1) >> 1; break; }
                        j += cnt; t += cnt; lim -= cnt;
                    }
                    ph = PH_STOP;
                    continue;
                }
                if (j < m && matches(sym(j))) { want = true; wsym = sym(j); wright = 1; base = cur; }
                else ph = PH_STOP;
            } else if (ph == PH_STOP) {
                // [x, j) is right-maximal, and left-maximal by construction: an SMEM
                if (j - x >= a.min_len) {
                    cg::coalesced_group g = cg::coalesced_threads();
                    unsigned long long at = 0;
                    if (g.thread_rank() == 0) at = atomicAdd(a.ctr + 3, (unsigned long long)g.size());
                    at = g.shfl(at, 0) + g.thread_rank();
                    if (at < a.cap) {
                        uint4* dst = reinterpret_cast<uint4*>(a.stage + at);
                        dst[0] = make_uint4(q, k, x, j);
                        dst[1] = make_uint4(cur.lb, cur.len, tg == kNone ? kNoSeq : tseq, tg == kNone ? 0u : tg - tbeg);
                    }
                    ++k;
                }
                tg = kNone;
                fresh = false;
                if (j >= m) { x = m; ph = PH_NEW; }
                else if (!matches(sym(j))) { x = j + 1; ph = PH_NEW; }
                else ph = PH_LEFT0;
            } else if (ph == PH_LEFT0) {
                want = true; wsym = sym(j); wright = 0; base = whole;
            } else {  // PH_LEFT: cur = cursor of Q[b:j+1]
                if (b > x + 1) {
                    const uint32_t c = sym(b - 1);
                    if (matches(c)) { want = true; wsym = c; wright = 0; base = cur; continue; }
                }
                x = b; ++j; ph = PH_RIGHT;
            }
        }
        if (!want) break;
        // ---- one bidirectional step ------------------------------------------------------------------------------------------
        const Cursor nx = extend_bi(ix, base, wsym, wright, look);
        ++ext;
        if (ph == PH_NEW) {
            if (nx.len) { cur = nx; j = x + 1; ph = PH_RIGHT; fresh = true; } else ++x;
        } else if (ph == PH_RIGHT) {
            if (nx.len) { cur = nx; ++j; } else ph = PH_STOP;
        } else if (ph == PH_LEFT0) {
            if (nx.len) { cur = nx; b = j; ph = PH_LEFT; } else { x = j + 1; ph = PH_NEW; }
        } else {
            if (nx.len) { cur = nx; --b; } else { x = b; ++j; ph = PH_RIGHT; }
        }
    }
    __syncwarp();
    ext = __reduce_add_sync(0xFFFFFFFFu, ext);
    look = __reduce_add_sync(0xFFFFFFFFu, look);
    lines = __reduce_add_sync(0xFFFFFFFFu, lines);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(a.ctr + 0, (unsigned long long)ext);
        atomicAdd(a.ctr + 1, (unsigned long long)look);
        atomicAdd(a.ctr + 2, (unsigned long long)lines);
    }
}

// staged records -> (qidx, begin) order: record k of query q goes to start[q] + k
__global__ void __launch_bounds__(256) smem_scatter_kernel(const SmemStage* __restrict__ stage, uint64_t count, const uint32_t* __restrict__ start,
                                                           uint32_t qidx_base, SmemRec* __restrict__ out, uint2* __restrict__ at) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    const SmemStage s = stage[i];
    const uint32_t d = __ldg(start + s.q) + s.k;
    out[d] = SmemRec{s.q + qidx_base, s.begin, s.end, s.lb, s.len};
    at[d] = make_uint2(s.seq, s.pos);
}

// SMEM records -> dense hit records of locate: record i becomes the rows [lb, lb + min(len, max_occ)), reported with qidx = i
__global__ void __launch_bounds__(256) smem_to_hits_kernel(const SmemRec* __restrict__ smems, uint64_t count, uint64_t max_occ,
                                                           HitRec* __restrict__ hits, uint32_t* __restrict__ lens) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i > count) return;
    if (i == count) { lens[i] = 0; return; }
    const SmemRec s = smems[i];
    const uint32_t len = (uint64_t)s.len < max_occ ? s.len : (uint32_t)max_occ;
    hits[i] = HitRec{(uint32_t)i, s.lb, 0u, len, s.end - s.begin, 0u};
    lens[i] = len;
}

int check_smem_index(const fmb_index* ix) {
    if (!ix->bidirectional) { set_error("SMEM search needs a bidirectional index (a unidirectional one has no right step)"); return FMB_EUNSUPPORTED; }
    if (!ix->first_symb) { set_error("SMEM search needs sequence borders: FMB_INDEX_NO_DELIM indices have none"); return FMB_EUNSUPPORTED; }
    return FMB_OK;
}

template <class OCC>
int launch_smem(const fmb_index* ix, const IndexView<OCC>& v, const SmemArgs& args, cudaStream_t st) {
    int per_sm = 0;
    FMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, smem_kernel<OCC>, 256, 0));
    const unsigned grid = std::max(1u, std::min<unsigned>(grid_for(args.nq, 256), (unsigned)(std::max(per_sm, 1) * ix->sm_count)));
    smem_kernel<OCC><<<grid, 256, 0, st>>>(v, args);
    FMB_CUDA(cudaGetLastError());
    note_launches(1);
    return FMB_OK;
}

}  // namespace
}  // namespace fmb

using namespace fmb;

extern "C" {

int fmb_search_smems(const fmb_index* ix, const fmb_queries* q, uint32_t min_len, fmb_results** out) {
    if (!ix || !q || !out) { set_error("NULL argument"); return FMB_EINVAL; }
    *out = nullptr;
    if (q->device != ix->device) { set_error("queries live on device %d, index on %d", q->device, ix->device); return FMB_EINVAL; }
    FMB_TRY(check_smem_index(ix));
    FMB_TRY(use_device(ix->device));
    cudaStream_t st = active_stream(ix);
    const uint64_t nq = q->nq;
    DevBuf<unsigned long long> ctr;
    DevBuf<uint32_t> counts;
    DevBuf<SmemStage> stage;
    FMB_TRY(ctr.alloc(8));
    FMB_TRY(counts.alloc(nq + 1));
    SmemArgs args{};
    args.qsym = q->symbols.p;
    args.qoff = q->offsets.p;
    args.qflags = q->flags.p;
    args.qpk = q->packed.p;
    args.nq = (uint32_t)nq;
    args.min_len = min_len;
    if (ix->bikmer.p) {
        args.bikmer = ix->bikmer.p;
        args.bikmer_k = ix->bikmer_k;
        args.bikmer_base = ix->dna ? 0u : ix->sigma - ix->first_symb;
    }
    if (ix->isa.p && q->packed.p && q->flags.p) {
        args.text32 = ix->text2.p;
        args.rowpos = ix->view_rowpos();
    }
    args.counts = counts.p;
    args.ctr = ctr.p;
    EventTimer whole(st);
    unsigned long long h_ctr[8] = {0};
    uint64_t cap = std::max<uint64_t>(uint64_t(1) << 20, 4 * nq);
    float search_ms = 0;
    // grow and retry: a second attempt runs with the exact number of records the first one found
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (stage.alloc(cap) != FMB_OK) {
            set_error("SMEM search: %llu records do not fit the device; split the query batch", (unsigned long long)cap);
            return FMB_EOVERFLOW;
        }
        args.stage = stage.p;
        args.cap = cap;
        FMB_CUDA(cudaMemsetAsync(ctr.p, 0, 8 * sizeof(unsigned long long), st));
        FMB_CUDA(cudaMemsetAsync(counts.p + nq, 0, sizeof(uint32_t), st));
        EventTimer tm(st);
        if (nq) {
            if (ix->dna) FMB_TRY(launch_smem(ix, ix->view_dna(), args, st));
            else FMB_TRY(launch_smem(ix, ix->view_gen(), args, st));
        }
        FMB_CUDA(cudaMemcpyAsync(h_ctr, ctr.p, sizeof h_ctr, cudaMemcpyDeviceToHost, st));
        search_ms = (float)tm.stop();
        if (h_ctr[3] <= cap) break;
        cap = h_ctr[3];
    }
    if (h_ctr[3] > cap) { set_error("SMEM search: %llu records do not fit the %llu reserved", h_ctr[3], (unsigned long long)cap); return FMB_EOVERFLOW; }
    if (h_ctr[3] >= 0xFFFFFFFFull) { set_error("SMEM search: %llu records; this build reports fewer than 2^32 per call -- split the batch", h_ctr[3]); return FMB_EOVERFLOW; }
    const uint64_t total = h_ctr[3];
    auto res = new fmb_results();
    res->device = ix->device;
    res->kind = 2;
    auto fail = [&](int rc) { delete res; return rc; };
    int rc;
    if ((rc = res->smems.alloc(total)) || (rc = res->at.alloc(total))) return fail(rc);
    if (total) {
        if ((rc = exclusive_sum_u32(counts.p, counts.p, nq + 1, st))) return fail(rc);
        smem_scatter_kernel<<<grid_for(total, 256), 256, 0, st>>>(stage.p, total, counts.p, (uint32_t)q->qidx_base, res->smems.p, res->at.p);
        note_launches(2);
    }
    res->stats.kernel_ms = whole.stop();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("SMEM search: %s", cudaGetErrorString(e)); return fail(FMB_ECUDA); }
    res->stats.main_kernel_ms = search_ms;
    res->stats.extensions = h_ctr[0];
    res->stats.occ_lookups = h_ctr[1];
    res->stats.line_requests = h_ctr[2];
    res->count = total;
    res->slots = total;
    *out = res;
    return FMB_OK;
}

int fmb_locate_smems(const fmb_index* ix, const fmb_results* smems, uint64_t max_occ, fmb_results** out) {
    if (!ix || !smems || !out) { set_error("NULL argument"); return FMB_EINVAL; }
    *out = nullptr;
    FMB_TRY(check_smem_index(ix));
    if (smems->kind != 2) { set_error("fmb_locate_smems needs an SMEM result set (kind 2), got kind %d", smems->kind); return FMB_EINVAL; }
    if (smems->device != ix->device) { set_error("results live on another device"); return FMB_EINVAL; }
    FMB_TRY(use_device(ix->device));
    cudaStream_t st = active_stream(ix);
    const uint64_t ns = smems->count;
    EventTimer whole(st);
    // the SMEMs as dense hit records of the existing locate (K4): record i, rows lb .. lb + min(len, max_occ) - 1, at = the text path's
    // (seq, pos) of single-row records
    fmb_results hits;
    hits.device = ix->device;
    hits.kind = 0;
    hits.dense = true;
    hits.slots = ns;
    hits.count = max_occ ? ns : 0;
    FMB_TRY(hits.hits.alloc(ns));
    FMB_TRY(hits.lens.alloc(ns + 1));
    FMB_TRY(hits.at.alloc(ns));
    smem_to_hits_kernel<<<grid_for(ns + 1, 256), 256, 0, st>>>(smems->smems.p, ns, max_occ, hits.hits.p, hits.lens.p);
    FMB_CUDA(cudaGetLastError());
    note_launches(1);
    if (ns) FMB_CUDA(cudaMemcpyAsync(hits.at.p, smems->at.p, ns * sizeof(uint2), cudaMemcpyDeviceToDevice, st));
    fmb_results* loc = nullptr;
    FMB_TRY(fmb_locate(ix, &hits, &loc));
    auto res = new fmb_results();
    res->device = ix->device;
    res->kind = 3;
    res->locs = std::move(loc->locs);
    res->count = res->slots = loc->count;
    res->stats = loc->stats;
    fmb_results_destroy(loc);
    int rc = res->smems.alloc(ns);
    if (rc) { delete res; return rc; }
    if (ns) {
        cudaError_t e = cudaMemcpyAsync(res->smems.p, smems->smems.p, ns * sizeof(SmemRec), cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) { delete res; set_error("locate SMEMs: %s", cudaGetErrorString(e)); return FMB_ECUDA; }
    }
    res->stats.kernel_ms = whole.stop();
    *out = res;
    return FMB_OK;
}

int fmb_results_fetch_smems(const fmb_results* r, fmb_smem* out, uint64_t capacity) {
    if (!r || (!out && r->count)) { set_error("NULL argument"); return FMB_EINVAL; }
    if (r->kind != 2) { set_error("result set holds no SMEMs (kind %d)", r->kind); return FMB_EINVAL; }
    if (capacity < r->count) { set_error("capacity %llu < %llu SMEMs", (unsigned long long)capacity, (unsigned long long)r->count); return FMB_EOVERFLOW; }
    FMB_TRY(use_device(r->device));
    std::vector<SmemRec> h(r->count);
    if (r->count) FMB_CUDA(cudaMemcpy(h.data(), r->smems.p, r->count * sizeof(SmemRec), cudaMemcpyDeviceToHost));
    for (uint64_t i = 0; i < r->count; ++i) out[i] = fmb_smem{h[i].qidx, h[i].begin, h[i].end, h[i].lb, h[i].len};
    return FMB_OK;
}

int fmb_results_fetch_smem_locs(const fmb_results* r, fmb_smem_loc* out, uint64_t capacity) {
    if (!r || (!out && r->count)) { set_error("NULL argument"); return FMB_EINVAL; }
    if (r->kind != 3) { set_error("result set holds no located SMEM rows (kind %d)", r->kind); return FMB_EINVAL; }
    if (capacity < r->count) { set_error("capacity %llu < %llu rows", (unsigned long long)capacity, (unsigned long long)r->count); return FMB_EOVERFLOW; }
    FMB_TRY(use_device(r->device));
    std::vector<LocRec> rows(r->count);
    std::vector<SmemRec> sm(r->smems.n);
    if (r->count) FMB_CUDA(cudaMemcpy(rows.data(), r->locs.p, r->count * sizeof(LocRec), cudaMemcpyDeviceToHost));
    if (r->count) FMB_CUDA(cudaMemcpy(sm.data(), r->smems.p, sm.size() * sizeof(SmemRec), cudaMemcpyDeviceToHost));
    for (uint64_t i = 0; i < r->count; ++i) {
        const SmemRec& s = sm[rows[i].qidx];
        out[i] = fmb_smem_loc{s.qidx, s.begin, s.end, rows[i].seq, rows[i].pos};
    }
    return FMB_OK;
}

}  // extern "C"
