// fmb_device.cuh -- device-side occurrence table ("String_c" of the reference, string/concepts.h:26-87) and
// cursor arithmetic (fmindex/BiFMIndexCursor.h:58-128, 180-190, 248-255) for sm_100a.
//
// Layout K1 (SURVEY.md §7 step 3, north_star subsystem 1)
// -------------------------------------------------------
// DNA layout (OccDna), sigma <= 5 (symbol 0 = delimiter, 1..4): one 32-byte block per 64 BWT rows
//     u32 cnt[4]   absolute number of symbols 1..4 in rows [0, 64*b)
//     u64 p0, p1   bit r of p0/p1 = low/high bit of (BWT[64*b + r] - 1); delimiter rows are coded like symbol 1
//   One rank / prefix_rank / all_ranks / symbol query = ONE aligned 32-byte sector, fetched with a single
//   LDG.E.256.  Delimiter rows (one per sequence) live in a sorted side list `delim_rows`.  The number of
//   delimiter rows before a block is implied by the block itself (64*b - sum(cnt)), so a correction only looks
//   at delim_rows[that index ...]; with a single sequence it is a register compare.
//
// Generic layout (OccGen), 5 < sigma <= 64: one block of `stride` bytes (multiple of 32) per 64 rows
//     u64 plane[B]        B = ceil(log2 sigma) bit planes of the symbols
//     u32 pc[sigma-1]     pc[c-1] = # symbols < c in rows [0, 64*b), c = 1..sigma-1   (exclusive prefix counts,
//                         the same quantity string/FlattenedBitvectors2L.h:226-239 keeps per block)
//   sigma = 21: 40 + 80 = 120 -> 128-byte blocks; a lookup touches the planes (2 sectors) + 1..2 count sectors.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace fmb {

typedef uint32_t row_t;   // this build: n < 2^32 - 64

__device__ __forceinline__ uint64_t low_mask(uint32_t off) {   // off in [0,63]
    return (uint64_t(1) << off) - 1;
}

// =========================================================================================================
// DNA layout
// =========================================================================================================
struct alignas(32) DnaBlock {
    uint32_t cnt[4];
    uint64_t p0, p1;
};
static_assert(sizeof(DnaBlock) == 32, "one sector");

struct OccDna {
    typedef DnaBlock Block;
    static constexpr bool kSymbolLoad = false;   // one load serves every symbol
    const DnaBlock* blocks;      // n/64 + 1 blocks
    const uint32_t* delim_rows;  // sorted rows holding symbol 0, padded with one 0xFFFFFFFF entry
    uint32_t n_delims;
    uint32_t delim0;             // delim_rows[0] (register copy for the single-sequence case)

    __device__ __forceinline__ DnaBlock load(uint32_t blk, uint32_t /*symb*/ = 0) const {
        DnaBlock b;
        uint32_t a0, a1, a2, a3, a4, a5, a6, a7;
        asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3), "=r"(a4), "=r"(a5), "=r"(a6), "=r"(a7)
                     : "l"(blocks + blk));
        b.cnt[0] = a0; b.cnt[1] = a1; b.cnt[2] = a2; b.cnt[3] = a3;
        b.p0 = (uint64_t)a4 | ((uint64_t)a5 << 32);
        b.p1 = (uint64_t)a6 | ((uint64_t)a7 << 32);
        return b;
    }

    // cnt[k] without dynamic indexing (a runtime index would push the block into local memory)
    static __device__ __forceinline__ uint32_t cnt_of(const DnaBlock& b, uint32_t k) {
        return (k & 2) ? ((k & 1) ? b.cnt[3] : b.cnt[2]) : ((k & 1) ? b.cnt[1] : b.cnt[0]);
    }
    // bit r set <=> row r of the block holds code k (k = symbol-1; delimiter rows alias k = 0)
    static __device__ __forceinline__ uint64_t match_mask(const DnaBlock& b, uint32_t k) {
        uint64_t m0 = (k & 1) ? b.p0 : ~b.p0;
        uint64_t m1 = (k & 2) ? b.p1 : ~b.p1;
        return m0 & m1;
    }
    // bit r set <=> code of row r is < k  (k in 0..4)
    static __device__ __forceinline__ uint64_t less_mask(const DnaBlock& b, uint32_t k) {
        uint64_t any = ~uint64_t(0);
        uint64_t m = 0;
        m = (k == 1) ? (~b.p1 & ~b.p0) : m;
        m = (k == 2) ? (~b.p1) : m;
        m = (k == 3) ? ~(b.p1 & b.p0) : m;
        m = (k >= 4) ? any : m;
        return m;
    }
    static __device__ __forceinline__ uint32_t delims_before_block(const DnaBlock& b, uint32_t blk) {
        return blk * 64u - (b.cnt[0] + b.cnt[1] + b.cnt[2] + b.cnt[3]);
    }
    // number of delimiter rows in [0,row); blk = row >> 6
    __device__ __forceinline__ uint32_t delims_below(const DnaBlock& b, row_t row) const {
        if (n_delims == 1) return delim0 < row ? 1u : 0u;
        uint32_t d = delims_before_block(b, row >> 6);
        while (__ldg(delim_rows + d) < row) ++d;     // padded with 0xFFFFFFFF: terminates
        return d;
    }
    // rank(row, symb): # rows < row with BWT == symb                            (string/concepts.h:52-56)
    __device__ __forceinline__ uint32_t rank(const DnaBlock& b, row_t row, uint32_t symb) const {
        if (symb == 0) return delims_below(b, row);
        uint32_t k = symb - 1;
        uint32_t r = cnt_of(b, k) + __popcll(match_mask(b, k) & low_mask(row & 63));
        if (k == 0) r -= delims_below(b, row) - delims_before_block(b, row >> 6);
        return r;
    }
    // prefix_rank(row, symb), symb in 0..sigma: # rows < row with BWT < symb    (string/concepts.h:58-64)
    __device__ __forceinline__ uint32_t prefix_rank(const DnaBlock& b, row_t row, uint32_t symb) const {
        if (symb == 0) return 0;
        if (symb == 1) return delims_below(b, row);
        uint32_t k = symb - 1;                        // k >= 1: delimiter rows alias code 0 < k, counted by the mask
        uint32_t r = delims_before_block(b, row >> 6);
#pragma unroll
        for (uint32_t j = 0; j < 4; ++j) r += (j < k) ? b.cnt[j] : 0u;
        return r + __popcll(less_mask(b, k) & low_mask(row & 63));
    }
    // symbol(row)                                                               (string/concepts.h:48-50)
    __device__ __forceinline__ uint32_t symbol(const DnaBlock& b, row_t row) const {
        uint32_t off = row & 63;
        uint32_t k = (uint32_t)((b.p0 >> off) & 1) | ((uint32_t)((b.p1 >> off) & 1) << 1);
        if (k == 0) {
            if (n_delims == 1) return delim0 == row ? 0u : 1u;
            uint32_t d = delims_below(b, row);
            if (__ldg(delim_rows + d) == row) return 0;
        }
        return k + 1;
    }
    // fused: rank(row,symb) and prefix_rank(row,symb) from one block
    __device__ __forceinline__ void rank_pr(const DnaBlock& b, row_t row, uint32_t symb, uint32_t& r, uint32_t& pr) const {
        r = rank(b, row, symb);
        pr = prefix_rank(b, row, symb);
    }
};

// =========================================================================================================
// DNA two-symbol layout (OccDna2): one 128-byte line per 128 BWT rows, resolved by a group of 4 lanes
// =========================================================================================================
// Why: ncu shows that every random 32-byte lookup moves a whole 128-byte DRAM line (profiles/r01_ncu_exact_v1.txt:
// dram__bytes_read = 116 B per lookup at 5.3 TB/s), and the request rate of random lines saturates at ~38 G/s
// whether 16, 32 or 128 bytes of the line are used (profiles/r01_gather_*.txt).  So a lookup should use the whole
// line it pays for: this block answers rank queries over PAIRS of symbols -- one line fetch advances a query by two
// symbols.  (The reference has the same idea as an experimental `KStep` path, search/SearchNoErrors.h:46-58.)
//
// pair code of row i = (y-1)*4 + (x-1) with y = T[SA[i]-1] (= BWT[i]) and x = T[SA[i]-2]; rows where x or y is the
// delimiter ("special" rows, two per sequence) are stored as code 0 and listed in a sorted side array.
// The line is four 32-byte quarters; quarter k (fetched by lane k of the group with one LDG.256):
//     u32 cnt[4]    absolute # rows before the block with code 4k .. 4k+3 (special rows count as code 0)
//     u32 plane[4]  bit r of plane[j] = bit j of the code of row 128*b + 32*k + r
// rank2(row, code) = sum over the 4 lanes of (popc(match(code) & rows-below-mask) + own counter) -> 2 SHFL.XOR.

// Where the suffix of a row starts in the text (fmb_index::view_rowpos, row_pos below), from the locate shortcut table in either of its
// forms: the suffix array (sa[row] = g of s0 0 s1 0 ..., its sequence through seq_of_block) or, without it, the shortcut word
// locrow[row] = sample index << step_bits | LF steps to that sample.
struct RowPosView {
    const uint32_t* sa;          // nullptr: the shortcut form
    const uint2* seq_of_block;
    const uint32_t* seq_start;   // start of every sequence (+ n); nullptr before the text check tables exist
    const uint32_t* locrow;
    const uint2* samples;
    uint32_t step_bits;
    uint32_t rate;               // text-regular sampling at this rate (a row's LF steps are pos % rate); 0: irregular
};

struct Occ2View {
    const uint4* lines;          // 8 uint4 per block; nullptr when the table was not built
    const uint32_t* specials;    // sorted special rows, padded with 0xFFFFFFFF
    uint32_t n_specials;
    uint32_t s0, s1;             // specials[0], specials[1] (register copies; single-sequence case)
    uint32_t C2[16];             // C2[code] = first row of the interval of the two-symbol pattern "x y"
    // k-mer table: (lb, len) of every pattern of kmer_k symbols over {1..4}; entry index = sum (s_p - 1) * 4^p with
    // s_0 the FIRST symbol of the pattern (the order of the 2-bit packed query stream).  Replaces the first kmer_k backward steps (the wide-interval phase, two
    // lines per step) by one lookup.  kmer_k = 0: no table.
    const uint2* kmer;
    uint32_t kmer_k;
    // LF^16 jump table: jump[row] = {LF^16(row), the 16 symbols preceding the suffix of `row` as 2-bit codes (symbol-1),
    // farthest symbol in the low bits = text order}; .x = 0xFFFFFFFF when one of the 16 symbols is a delimiter.  Once an interval is a
    // single row, 16 backward steps are one 8-byte lookup: compare the 32-bit symbol word with the query, follow .x.
    const uint2* jump;
    const uint2* jump4;          // the same with LF^4 and four symbols (8 bits): tails shorter than 16 symbols
    // jump_wide != 0: `jump` holds 16-byte entries {LF^16(row), symbols 1..16, LF^32(row), symbols 17..32} -- one lookup serves a
    // 16- or a 32-symbol jump (.z = 0xFFFFFFFF when one of symbols 17..32 is a delimiter)
    uint32_t jump_wide;
    // text check (fmb_index::isa / text2; isa == nullptr: none): a single-row interval r with pos query symbols left lies at text
    // position g = row_pos(r).g; the read can only be the text [g - pos, g) of g's sequence, compared with the query a 128-byte line
    // (512 symbols) at a time, and its row is isa[g - pos]
    const uint32_t* isa;
    const uint32_t* text32;      // 16 symbols per word, 32 words per 128-byte line
    RowPosView rowpos;
};
constexpr uint32_t kJumpInvalid = 0xFFFFFFFFu;
constexpr uint32_t kNoSeq = 0xFFFFFFFFu;      // fmb_results::at of a hit the text check did not find

// Sequence of text position g of s0 0 s1 0 ... (fmb_index::seq_of_block): per 4096-symbol block b, {s | inner << 31, seq_start[s]}
// with s the sequence holding the block's first symbol and inner set when another sequence starts inside the block.  Without such a
// start the answer is the one entry (one cached load: the table is n / 512 bytes); else a binary search of seq_start between s and the
// sequence of the next block's first symbol.  `lines` counts the loads.
struct SeqStart {
    uint32_t seq, start;
};
__device__ __forceinline__ SeqStart seq_of(const uint2* __restrict__ blocks, const uint32_t* __restrict__ seq_start, uint32_t g, uint32_t& lines) {
    const uint2 e = __ldg(blocks + (g >> 12));
    lines += 1;
    SeqStart r{e.x & 0x7FFFFFFFu, e.y};
    if (e.x >> 31) {
        uint32_t hi = (__ldg(&blocks[(g >> 12) + 1].x) & 0x7FFFFFFFu) + 1;      // seq_start[hi] > g (seq_start[nseq] = n)
        lines += 1;
        while (hi - r.seq > 1) {
            const uint32_t mid = (r.seq + hi) >> 1, v = __ldg(seq_start + mid);
            lines += 1;
            if (v <= g) r = SeqStart{mid, v}; else hi = mid;
        }
    }
    return r;
}

// Text position of the suffix of `row`: its sequence, the position in it and the LF steps the walk to its sample takes; with kText also
// the global position g and the sequence's start (the shortcut form then reads seq_start, which exists with the text check tables).
// `lines` counts the loads of kText callers: 1 + seq_of's for the suffix array, 3 for the shortcut.
struct RowPos {
    uint32_t seq, pos, steps, g, start;
};
template <bool kText>
__device__ __forceinline__ RowPos row_pos(const RowPosView& v, row_t row, uint32_t& lines) {
    RowPos r;
    if (v.sa) {
        r.g = __ldg(v.sa + row);
        lines += 1;
        const SeqStart ss = seq_of(v.seq_of_block, v.seq_start, r.g, lines);
        r.seq = ss.seq;
        r.start = ss.start;
        r.pos = r.g - ss.start;
        r.steps = r.pos % v.rate;
    } else {
        const uint32_t w = __ldg(v.locrow + row);
        const uint2 smp = __ldg(v.samples + (w >> v.step_bits));
        r.steps = w & ((1u << v.step_bits) - 1u);
        r.seq = smp.x;
        r.pos = smp.y + r.steps;
        lines += 2;
        if (kText) {
            r.start = __ldg(v.seq_start + smp.x);
            r.g = r.start + r.pos;
            lines += 1;
        }
    }
    return r;
}

struct Quarter {
    uint32_t cnt[4];
    uint32_t plane[4];
};

__device__ __forceinline__ Quarter load_quarter(const Occ2View& o, uint32_t blk, uint32_t sub) {
    Quarter q;
    const uint4* p = o.lines + ((size_t)blk * 8 + sub * 2);
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(q.cnt[0]), "=r"(q.cnt[1]), "=r"(q.cnt[2]), "=r"(q.cnt[3]), "=r"(q.plane[0]), "=r"(q.plane[1]),
                   "=r"(q.plane[2]), "=r"(q.plane[3])
                 : "l"(p));
    return q;
}
// this lane's share of rank2(row, code): rows of quarter `sub` below `row` that hold `code`, plus the block counter
// when this quarter owns it
__device__ __forceinline__ uint32_t rank2_part(const Quarter& q, uint32_t sub, uint32_t row, uint32_t code) {
    uint32_t m = ((code & 1) ? q.plane[0] : ~q.plane[0]) & ((code & 2) ? q.plane[1] : ~q.plane[1]) &
                 ((code & 4) ? q.plane[2] : ~q.plane[2]) & ((code & 8) ? q.plane[3] : ~q.plane[3]);
    int rel = (int)(row & 127u) - (int)(sub * 32u);
    uint32_t mask = rel <= 0 ? 0u : (rel >= 32 ? 0xFFFFFFFFu : ((1u << rel) - 1u));
    uint32_t c = (code & 2) ? ((code & 1) ? q.cnt[3] : q.cnt[2]) : ((code & 1) ? q.cnt[1] : q.cnt[0]);
    return __popc(m & mask) + (((code >> 2) == sub) ? c : 0u);
}
// # special rows < row (they are stored as code 0 and must not count as the pair "1 1")
__device__ __forceinline__ uint32_t specials_below(const Occ2View& o, uint32_t row) {
    if (o.n_specials <= 2) return (o.s0 < row ? 1u : 0u) + (o.s1 < row ? 1u : 0u);
    uint32_t lo = 0, hi = o.n_specials;
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(o.specials + mid) < row) lo = mid + 1; else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ uint32_t group_sum4(uint32_t v, uint32_t gmask) {
    v += __shfl_xor_sync(gmask, v, 1);
    v += __shfl_xor_sync(gmask, v, 2);
    return v;
}

// =========================================================================================================
// generic layout
// =========================================================================================================
struct GenBlock {
    uint64_t plane[6];
    uint32_t pc_lo, pc_hi;       // pc[symb-1] (0 for symb 0) and pc[symb] (block start for symb = sigma-1)
};

struct OccGen {
    typedef GenBlock Block;
    static constexpr bool kSymbolLoad = true;    // a loaded block carries the counts of ONE symbol
    const uint8_t* blocks;
    uint32_t stride;             // bytes per block (multiple of 32)
    uint32_t planes;             // B
    uint32_t sigma;

    // the block is loaded for ONE symbol: planes + the two prefix counts that bracket it
    __device__ __forceinline__ GenBlock load(uint32_t blk, uint32_t symb) const {
        GenBlock b;
        const uint8_t* p = blocks + (size_t)blk * stride;
        const ulonglong2* pp = reinterpret_cast<const ulonglong2*>(p);
#pragma unroll
        for (uint32_t j = 0; j < 3; ++j) {
            if (2 * j < planes) {
                ulonglong2 v = __ldg(pp + j);
                b.plane[2 * j] = v.x;
                b.plane[2 * j + 1] = v.y;   // may hold count words when planes is odd; masked by `planes` later
            } else {
                b.plane[2 * j] = b.plane[2 * j + 1] = 0;
            }
        }
        const uint32_t* pc = reinterpret_cast<const uint32_t*>(p + 8 * planes);
        b.pc_lo = symb == 0 ? 0u : __ldg(pc + symb - 1);
        b.pc_hi = symb + 1 >= sigma ? blk * 64u : __ldg(pc + symb);
        return b;
    }
    __device__ __forceinline__ uint64_t match_mask(const GenBlock& b, uint32_t symb) const {
        uint64_t m = ~uint64_t(0);
#pragma unroll
        for (uint32_t j = 0; j < 6; ++j)
            if (j < planes) m &= ((symb >> j) & 1) ? b.plane[j] : ~b.plane[j];
        return m;
    }
    // rows whose symbol is < symb: classic bit-serial comparison from the top plane down
    __device__ __forceinline__ uint64_t less_mask(const GenBlock& b, uint32_t symb) const {
        uint64_t lt = 0, eq = ~uint64_t(0);
#pragma unroll
        for (int j = 5; j >= 0; --j) {
            if ((uint32_t)j < planes) {
                uint64_t pj = b.plane[j];
                if ((symb >> j) & 1) { lt |= eq & ~pj; eq &= pj; }
                else { eq &= ~pj; }
            }
        }
        return lt;
    }
    __device__ __forceinline__ uint32_t rank(const GenBlock& b, row_t row, uint32_t symb) const {
        return (b.pc_hi - b.pc_lo) + __popcll(match_mask(b, symb) & low_mask(row & 63));
    }
    __device__ __forceinline__ uint32_t prefix_rank(const GenBlock& b, row_t row, uint32_t symb) const {
        return b.pc_lo + __popcll(less_mask(b, symb) & low_mask(row & 63));
    }
    __device__ __forceinline__ void rank_pr(const GenBlock& b, row_t row, uint32_t symb, uint32_t& r, uint32_t& pr) const {
        r = rank(b, row, symb);
        pr = prefix_rank(b, row, symb);
    }
    __device__ __forceinline__ uint32_t symbol(const GenBlock& b, row_t row) const {
        uint32_t off = row & 63, s = 0;
#pragma unroll
        for (uint32_t j = 0; j < 6; ++j)
            if (j < planes) s |= (uint32_t)((b.plane[j] >> off) & 1) << j;
        return s;
    }
};

// =========================================================================================================
// device view of a whole index and the cursor steps
// =========================================================================================================
template <class OCC>
struct IndexView {
    OCC occ[2];             // [0] = bwt, [1] = bwtRev (blocks == nullptr when unidirectional)
    uint32_t C[65];         // C[s] = # symbols < s in the BWT, s = 0..sigma      (utils.h:200-206)
    row_t n;                // rows
    uint32_t sigma;
    uint32_t first_symb;    // FirstSymb of the index (fmindex/BiFMIndex.h:26): 1 = symbol 0 is the sequence delimiter, 0 = NoDelim
    // sampled suffix array (suffixarray/SparseArray.h:63-70): per 64 rows {u64 marker bits, u32 samples before}
    const uint4* marks;     // .x,.y = marker bits (low, high word), .z = number of samples before the word
    const uint2* samples;   // .x = seqId, .y = pos
    // locate blocks (DNA layout only): per 64 rows one 64-byte record = {DnaBlock (32 B), marker bits u64, samples before
    // u32, pad} so that one LF step of locate touches ONE line instead of two (occ block + marker word); a lane pair
    // fetches the two 32-byte halves with one request.  nullptr when not built.
    const uint4* locblocks;
};

struct Cursor {             // BiFMIndexCursor{lb, lbRev, len, steps}, fmindex/BiFMIndexCursor.h:22-37
    row_t lb, lb_rev, len;
    uint32_t steps;
};

// LeftBiFMIndexCursor::extendLeft(symb) / FMIndexCursor::extendLeft(symb)
// (fmindex/BiFMIndexCursor.h:248-255, fmindex/FMIndexCursor.h:33-37):
//     lb' = C[c] + rank(lb,c),  len' = rank(lb+len,c) - rank(lb,c)
// `lookups` counts occ blocks fetched (1 when both ends share a block, else 2) -- SURVEY.md §8(d) work unit.
template <class OCC>
__device__ __forceinline__ void extend_left_uni(const IndexView<OCC>& ix, row_t& lb, row_t& len, uint32_t symb, uint32_t& lookups) {
    const OCC& occ = ix.occ[0];
    row_t hi = lb + len;
    uint32_t b0 = lb >> 6, b1 = hi >> 6;
    typename OCC::Block blk0 = occ.load(b0, symb);
    uint32_t r0, r1;
    if (b1 == b0) {
        r0 = occ.rank(blk0, lb, symb);
        r1 = occ.rank(blk0, hi, symb);
        lookups += 1;
    } else {
        typename OCC::Block blk1 = occ.load(b1, symb);
        r0 = occ.rank(blk0, lb, symb);
        r1 = occ.rank(blk1, hi, symb);
        lookups += 2;
    }
    lb = ix.C[symb] + r0;
    len = r1 - r0;
}

// BiFMIndexCursor::extendLeft(symb) (:113-120) when right == 0, extendRight(symb) (:121-128) when right == 1.
template <class OCC>
__device__ __forceinline__ Cursor extend_bi(const IndexView<OCC>& ix, const Cursor& c, uint32_t symb, int right, uint32_t& lookups) {
    const OCC& occ = ix.occ[right];
    row_t lo = right ? c.lb_rev : c.lb;
    row_t hi = lo + c.len;
    uint32_t b0 = lo >> 6, b1 = hi >> 6;
    typename OCC::Block blk0 = occ.load(b0, symb);
    uint32_t r0, p0, r1, p1;
    if (b1 == b0) {
        occ.rank_pr(blk0, lo, symb, r0, p0);
        occ.rank_pr(blk0, hi, symb, r1, p1);
        lookups += 1;
    } else {
        typename OCC::Block blk1 = occ.load(b1, symb);
        occ.rank_pr(blk0, lo, symb, r0, p0);
        occ.rank_pr(blk1, hi, symb, r1, p1);
        lookups += 2;
    }
    Cursor o;
    row_t same = ix.C[symb] + r0;
    row_t other = (right ? c.lb : c.lb_rev) + (p1 - p0);
    o.lb = right ? other : same;
    o.lb_rev = right ? same : other;
    o.len = r1 - r0;
    o.steps = c.steps + 1;
    return o;
}

// One LF step (fmindex/BiFMIndex.h:177-202): c = BWT[row], row' = C[c] + rank(row, c).  b = the occ block of row, loaded for symbol 0.
template <class OCC>
__device__ __forceinline__ row_t lf_step(const IndexView<OCC>& ix, typename OCC::Block b, row_t row, uint32_t& c) {
    const OCC& occ = ix.occ[0];
    c = occ.symbol(b, row);
    if (OCC::kSymbolLoad) b = occ.load(row >> 6, c);
    return ix.C[c] + occ.rank(b, row, c);
}

// LF walk of one thread from `row` to the nearest sampled row: the sample's index (adding the LF steps to `steps`), or kNoSample after
// more than `limit` steps.  The marker word and the occ block of a row are independent loads and are issued together.
constexpr uint32_t kNoSample = 0xFFFFFFFFu;
template <class OCC>
__device__ __forceinline__ uint32_t walk_to_sample(const IndexView<OCC>& ix, row_t row, uint32_t& steps, uint32_t limit = 0xFFFFFFFFu) {
    for (;;) {
        const uint4 m = __ldg(ix.marks + (row >> 6));
        const typename OCC::Block b = ix.occ[0].load(row >> 6, 0);
        const uint64_t bits = (uint64_t)m.x | ((uint64_t)m.y << 32);
        const uint32_t o = row & 63;
        if ((bits >> o) & 1) return m.z + __popcll(bits & low_mask(o));
        uint32_t c;
        row = lf_step(ix, b, row, c);
        if (++steps > limit) return kNoSample;
    }
}

// Work counters: one global atomic per BLOCK and counter.  (One per warp meant > 10^6 same-address atomics per launch, which
// serialise in one L2 slice and cost more than the kernel's real work: locate went from 1.4 ms to the time of its loads.)
// Every thread of the block must call this (it contains __syncthreads).
__device__ __forceinline__ void block_count2(unsigned long long* counters, int slot_a, uint32_t a, int slot_b, uint32_t b) {
    __shared__ unsigned int s_cnt[2];
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xFFFFFFFFu, a, o);
        b += __shfl_xor_sync(0xFFFFFFFFu, b, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (a) atomicAdd(&s_cnt[0], a);
        if (b) atomicAdd(&s_cnt[1], b);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_cnt[0]) atomicAdd(counters + slot_a, (unsigned long long)s_cnt[0]);
        if (slot_b >= 0 && s_cnt[1]) atomicAdd(counters + slot_b, (unsigned long long)s_cnt[1]);
    }
}

// the same for three counters, the third one 64 bits wide (sum of interval lengths)
__device__ __forceinline__ void block_count3(unsigned long long* counters, int slot_a, uint32_t a, int slot_b, uint32_t b, int slot_c, unsigned long long c) {
    __shared__ unsigned int s_cnt[2];
    __shared__ unsigned long long s_cnt64;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    if (threadIdx.x == 2) s_cnt64 = 0;
    __syncthreads();
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xFFFFFFFFu, a, o);
        b += __shfl_xor_sync(0xFFFFFFFFu, b, o);
        c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (a) atomicAdd(&s_cnt[0], a);
        if (b) atomicAdd(&s_cnt[1], b);
        if (c) atomicAdd(&s_cnt64, c);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_cnt[0]) atomicAdd(counters + slot_a, (unsigned long long)s_cnt[0]);
        if (s_cnt[1]) atomicAdd(counters + slot_b, (unsigned long long)s_cnt[1]);
        if (s_cnt64) atomicAdd(counters + slot_c, s_cnt64);
    }
}

}  // namespace fmb
