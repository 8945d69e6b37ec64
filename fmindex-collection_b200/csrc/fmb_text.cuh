// fmb_text.cuh -- K3b: k-error search (edit and Hamming distance) on single-row intervals, decided on the TEXT instead of the index.
//
// Once the interval of a search is a single row, the search walks one fixed text: the row after t more symbols is LF^t(row) and
// the symbols it meets are the entries of jump[row], jump[LF^16(row)], ... (16 symbols per 8-byte lookup; LF^4 with byte symbols
// for the generic layout).  The whole subtree of such a node -- as long as the search keeps its direction -- is therefore a
// function of (text window, query, scheme): the node state machine of search_ng26 (search_next_pos / search_next_dir_single /
// search_next_dir_no_errors, search/SearchNg26.h:119-141, 225-365) is run here on the window symbols held in shared memory, with a
// private depth-first stack per lane, and the index is touched only to fetch the window (one lookup per 16 symbols) and to compute
// the rows of the few paths that survive.  What leaves the walk of an item is a hand-over (an item again):
//   * a child whose position advance ends the last part of the direction run (the search turns around or ends): the child exactly
//     as search_next_dir_single creates it, advance pending                                                    ("turn" items)
//   * an error-free stretch that ends a part the same way: the state search_next_dir_no_errors leaves (:241-249)
//   * a node at the end of the window (144 symbols, a delimiter ahead, or the private stack full): the node as it is ("continue")
//   * an item whose row has no usable window at all (delimiter within the next 16 symbols): the item itself, flagged `notext`
// A hand-over that ends the search is a leaf and is reported here; the others are single rows again -- text class -- and go straight
// to the text list of the next pass (SchemeOut::text_next); only `notext` items (and error-free stretches of the generic layout) go
// to the overflow list, i.e. to the frontier kernel (scheme_search_kernel), which expands them on the index.  Results are identical
// by construction: this is the same state machine on the same symbols; fmb_stats.extensions still equals the oracle's count (one per
// node visit, one per symbol of an error-free stretch).
//
// Work distribution: one item per LANE, in a flat loop -- every iteration each lane pops one node of its private stack (or takes its
// next item when the stack is empty) -- so that the lanes of a warp always execute the same loop body although their items need
// different numbers of node visits.
#pragma once
#include "fmb_scheme.cuh"

namespace fmb {

constexpr int kTextWords = 9;        // window words per lane: 144 symbols (2-bit codes) / 36 symbols (bytes)
constexpr int kTextQWords = 10;      // query words per lane, walking order: 160 / 40 symbols
constexpr int kTextStage = 64;       // staged items (and hits) per warp before they are flushed to the global lists (flushed at 32)
constexpr int kTextStack = 16;       // private depth-first stack (packed nodes)
#ifndef FMB_TEXT_MINB
#define FMB_TEXT_MINB 4
#endif

struct TNode {             // one pending node, "ready to expand" (the position advance already applied)
    uint32_t m;            // text symbols consumed since the item started: the node looks at window symbol m
    uint32_t c;            // query symbols consumed since the item started
    uint32_t part, pev, e;
    uint32_t T;            // info of the walking side (INFO_*)
    uint32_t lastRank, lastQRank;
    uint32_t noerr;        // inside the error-free loop
    uint32_t kind;         // TN_*: what happens to the node
};
// TN_EXPAND: a node of the private stack.  The other kinds are requests to hand the node to the frontier kernel:
// TN_TURN = a child of search_next_dir_single whose pending position advance ends the direction run (mode POS, NextPos 1),
// TN_NEXT = the state search_next_dir_no_errors leaves at such a part end (mode NEXT), TN_CONT = the node as it is (window end)
enum : uint32_t { TN_EXPAND = 0, TN_TURN = 1, TN_NEXT = 2, TN_CONT = 3 };
// kinds of the queued comparisons along a diagonal: LC_VISIT = a node without errors left (its own visit, then error free),
// LC_RUN = an error-free stretch, LC_SKIP = the matching stretch of a path at its last error level, LC_BULK2 = the matching stretch of
// a path with two errors left (its deletion / insertion subtrees are evaluated sixteen positions at a time)
enum : uint32_t { LC_VISIT = 0, LC_RUN = 1, LC_SKIP = 2, LC_BULK2 = 3 };
__device__ __forceinline__ unsigned long long tnode_pack(const TNode& s) {
    // m:8 c:8 part:5 pev:16 e:4 T:2 lastRank:8 lastQRank:8 noerr:1 kind:2
    return (unsigned long long)s.m | ((unsigned long long)s.c << 8) | ((unsigned long long)s.part << 16) | ((unsigned long long)s.pev << 21) |
           ((unsigned long long)s.e << 37) | ((unsigned long long)s.T << 41) | ((unsigned long long)s.lastRank << 43) |
           ((unsigned long long)s.lastQRank << 51) | ((unsigned long long)s.noerr << 59) | ((unsigned long long)s.kind << 60);
}
__device__ __forceinline__ TNode tnode_unpack(unsigned long long v) {
    TNode s;
    s.m = v & 255; s.c = (v >> 8) & 255; s.part = (v >> 16) & 31; s.pev = (v >> 21) & 0xFFFF; s.e = (v >> 37) & 15;
    s.T = (v >> 41) & 3; s.lastRank = (v >> 43) & 255; s.lastQRank = (v >> 51) & 255; s.noerr = (v >> 59) & 1; s.kind = (v >> 60) & 3;
    return s;
}
static_assert(kTextWords * 16 <= 255 && kTextQWords * 16 <= 255, "window / query positions are 8-bit fields of a packed node");

// reverses the order of the sixteen 2-bit fields of a word
__device__ __forceinline__ uint32_t rev2(uint32_t w) {
    w = __brev(w);
    return ((w & 0xAAAAAAAAu) >> 1) | ((w & 0x55555555u) << 1);
}

// a hit in the slot of an item (the warp stage of scheme_text_kernel holds both): meta = kHitMark cannot be an item (mode 3 does not exist)
constexpr uint32_t kHitMark = 0xFFFFFFFFu;
__device__ __forceinline__ Item item_of_hit(const HitRec& h) {
    Item it;
    it.lb = h.lb; it.lb_rev = h.lb_rev; it.len = h.len; it.qidx = h.qidx; it.qpos = h.steps; it.pev_steps = h.e; it.meta = kHitMark; it.side = 0;
    return it;
}
__device__ __forceinline__ HitRec hit_of_item(const Item& it) {
    HitRec h;
    h.qidx = it.qidx; h.lb = it.lb; h.lb_rev = it.lb_rev; h.len = it.len; h.steps = it.qpos; h.e = it.pev_steps;
    return h;
}

// Edit distance, TWO errors left, inside the part, after a match (2-bit symbols).  At a matching position c (text position m) the
// node's subtrees other than its match child are small and have a fixed shape (search_next_dir_single, SearchNg26.h:251-365):
//   deletion child D1 (m+1, c):  its symbol equals q[c]  -> one more deletion child, which dies                        (2 visits)
//                                else substitution S2 (m+2, c+1) and deletion D2 (m+2, c), both error free from there
//   insertion child I1 (m, c+1): q[c+1] != q[c]         -> substitution S2' (m+1, c+2), error free
//                                always                  -> insertion I2 (m, c+2), error free, its first match needs q[c+2] != q[c+1]
// so per position: 5 visits + [w[m+1] != q[c]] (1 + run S2 + run D2) + [q[c+1] != q[c]] (1 + run S2') + run I2, where an error-free path
// that matches r >= 1 symbols and then fails costs r + 1 extensions.  The four runs lie on the diagonals +1, +2, -1, -2 of the
// alignment: their match masks are XORs of shifted window / query words (one bit per position, at the even bits of a 64-bit mask),
// the run lengths come from iterated AND-shift.  Positions where a run goes on for kLook symbols -- or reaches the end of the part,
// where it may survive -- are not decided here: they are returned in `slow` (their own visit is counted; the caller pushes their two
// children).  Returns the extensions of the block [c0, c0 + nb); nb = 0: nothing decided.
// sw / sq: the lane's window / query words ([word][thread] layout), have_syms: window symbols fetched (>= m0 + min(pev0, 32) + 2).
__device__ __noinline__ uint32_t bulk2_eval(const uint32_t* sw, const uint32_t* sq, uint32_t tid, uint32_t have_syms, uint32_t m0, uint32_t c0, uint32_t pev0,
                                            uint32_t& nb_out, unsigned long long& slow_out) {
    constexpr uint32_t kLook = 8;
    constexpr unsigned long long EVEN = 0x5555555555555555ull;
    constexpr uint32_t QCAP = kTextQWords * 16;
    auto wword = [&](uint32_t m) -> uint32_t { return __funnelshift_r(sw[(m / 16) * 256 + tid], sw[(m / 16 + 1) * 256 + tid], 2 * (m % 16)); };
    auto qword = [&](uint32_t c) -> uint32_t { return __funnelshift_r(sq[(c / 16) * 256 + tid], sq[(c / 16 + 1) * 256 + tid], 2 * (c % 16)); };
    auto eq32 = [&](uint32_t ma, uint32_t ca) -> uint32_t { const uint32_t x = wword(ma) ^ qword(ca); return ~(x | (x >> 1)) & 0x55555555u; };
    auto eq64 = [&](uint32_t ma, uint32_t ca) -> unsigned long long {
        const unsigned long long lo = eq32(ma, ca);
        const unsigned long long hi = (ma + 16 < have_syms && ca + 32 <= QCAP) ? eq32(ma + 16, ca + 16) : 0u;
        return lo | (hi << 32);
    };
    nb_out = 0;
    slow_out = 0;
    const unsigned long long M0 = eq64(m0, c0);
    const unsigned long long miss = ~M0 & EVEN;
    uint32_t nb = miss ? (uint32_t)(__ffsll((long long)miss) - 1) / 2u : 32u;      // leading matches on the main diagonal
    nb = nb < 16u ? nb : 16u;
    nb = nb < pev0 - 3 ? nb : pev0 - 3;                                             // every position of the block keeps >= 4 symbols of the part
    if (nb == 0) return 0;
    const unsigned long long end0 = pev0 >= 32 ? 0ull : (EVEN << (2 * pev0));      // positions beyond the part: runs that get there stay "alive"
    const unsigned long long end2 = pev0 - 2 >= 32 ? 0ull : (EVEN << (2 * (pev0 - 2)));
    const unsigned long long E1 = eq64(m0 + 1, c0) | end0;                          // w[m+1+i] == q[c+i]
    const unsigned long long E2 = eq64(m0 + 2, c0) | end0;                          // w[m+2+i] == q[c+i]
    const unsigned long long N1 = eq64(m0 + 1, c0 + 2) | end2;                      // w[m+1+i] == q[c+2+i]
    const unsigned long long N2 = eq64(m0, c0 + 2) | end2;                          // w[m+i]   == q[c+2+i]
    unsigned long long F;                                                            // q[c+1+i] == q[c+i]
    {
        const uint32_t x0 = qword(c0 + 1) ^ qword(c0);
        const uint32_t x1 = (c0 + 33 <= QCAP) ? (qword(c0 + 17) ^ qword(c0 + 16)) : 0xFFFFFFFFu;
        F = (unsigned long long)(~(x0 | (x0 >> 1)) & 0x55555555u) | ((unsigned long long)(~(x1 | (x1 >> 1)) & 0x55555555u) << 32);
    }
    const unsigned long long BM0 = ((1ull << (2 * nb)) - 1) & EVEN;
    unsigned long long BM = BM0;
    uint32_t total = 0;
    for (int pass = 0; pass < 2; ++pass) {
        const unsigned long long A = ~E1 & BM, B = ~F & BM;
        unsigned long long U = 0, T;
        total = 5 * (uint32_t)__popcll(BM) + (uint32_t)__popcll(A) + (uint32_t)__popcll(B);
        T = A & (E1 >> 2);                                                           // S2: diagonal +1 from c+1
        total += 2 * (uint32_t)__popcll(T);
#pragma unroll 1
        for (uint32_t t = 1; t < kLook; ++t) { T &= E1 >> (2 * (1 + t)); total += (uint32_t)__popcll(T); }
        U |= T;
        T = A & E2;                                                                  // D2: diagonal +2 from c
        total += 2 * (uint32_t)__popcll(T);
#pragma unroll 1
        for (uint32_t t = 1; t < kLook; ++t) { T &= E2 >> (2 * t); total += (uint32_t)__popcll(T); }
        U |= T;
        T = B & N1;                                                                  // S2': diagonal -1 from c+2
        total += 2 * (uint32_t)__popcll(T);
#pragma unroll 1
        for (uint32_t t = 1; t < kLook; ++t) { T &= N1 >> (2 * t); total += (uint32_t)__popcll(T); }
        U |= T;
        T = BM & N2 & ~(F >> 2);                                                     // I2: diagonal -2 from c+2, first match needs q[c+2] != q[c+1]
        total += 2 * (uint32_t)__popcll(T);
#pragma unroll 1
        for (uint32_t t = 1; t < kLook; ++t) { T &= N2 >> (2 * t); total += (uint32_t)__popcll(T); }
        U |= T;
        if (U == 0) break;
        if (pass == 1 || __popcll(U) > 2) return 0;            // too many undecided positions: the caller walks this stretch node by node
        BM &= ~U;                                               // undecided positions: their children are expanded one by one
    }
    const unsigned long long slow = BM0 & ~BM;
    nb_out = nb;
    slow_out = slow;
    return total + (uint32_t)__popcll(slow);                    // (the undecided positions' own visits; their children count themselves)
}

template <class OCC, bool EDIT, bool PSEUDO>
__global__ void __launch_bounds__(256, FMB_TEXT_MINB) scheme_text_kernel(const __grid_constant__ IndexView<OCC> ix, const __grid_constant__ SchemeParams sp,
                                                                         const uint8_t* __restrict__ qsym, const uint64_t* __restrict__ qoff,
                                                                         const __grid_constant__ JumpView jv, const Item* __restrict__ items, uint64_t n_items,
                                                                         const __grid_constant__ SchemeOut out) {
    constexpr bool BYTES = OCC::kSymbolLoad;
    constexpr uint32_t B = BYTES ? 8u : 2u;              // bits per symbol
    constexpr uint32_t SPW = 32u / B;                     // symbols per word
    constexpr uint32_t SM = (1u << B) - 1u;
    constexpr uint32_t WCAP = kTextWords * SPW;           // symbols per window
    constexpr uint32_t QCAP = kTextQWords * SPW;          // query symbols per item

    __shared__ uint32_t sw[(kTextWords + 1) * 256];      // [word][thread]: window symbols in walking order, one zero word behind
    __shared__ uint32_t sq[(kTextQWords + 1) * 256];     // [word][thread]: query symbols in walking order
    __shared__ Item stage[8][kTextStage];                // hand-overs AND hits (a hit travels as an item with meta = kHitMark) of a warp
    __shared__ uint32_t stage_cnt[8];

    const uint32_t tid = threadIdx.x;
    const uint32_t lane = tid & 31, warp = tid >> 5;
    const uint32_t np = sp.n_parts;
    if (lane == 0) stage_cnt[warp] = 0;
    __syncwarp();

    unsigned long long stk[kTextStack];
    uint32_t rows[kTextWords + 1];
    int top = 0;
    uint32_t n_ext = 0, n_phys = 0;
    uint64_t next_item = blockIdx.x * (uint64_t)blockDim.x + tid;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;

    // per item
    Item it0;                      // the entry state (position advance applied, direction decided), mode POS / NextPos 0
    uint32_t R = 0, search = 0, have = 0, q_limit = 0;
    bool closed = false;

    auto dir_of = [&](uint32_t part) -> uint32_t { return (sp.pi[search][part - 1] < sp.pi[search][part]) ? 1u : 0u; };
    auto stage_emit = [&](const Item& it) {
        const uint32_t slot = atomicAdd(&stage_cnt[warp], 1u);
        if (slot < (uint32_t)kTextStage) {
            stage[warp][slot] = it;
        } else {
            atomicSub(&stage_cnt[warp], 1u);
            if (it.meta == kHitMark) {
                const unsigned long long g = atomicAdd(out.hit_count, 1ull);
                atomicAdd(out.row_count, 1ull);
                if (g < out.hit_capacity) out.hits[g] = hit_of_item(it);
            } else {
                const unsigned long long g = atomicAdd(out.overflow_count, 1ull);
                if (g < out.overflow_capacity) out.overflow[g] = it;
            }
        }
    };
    // one LF step of a single row in direction R
    auto lf1 = [&](uint32_t row) -> uint32_t {
        const OCC& occ = ix.occ[R];
        typename OCC::Block b = occ.load(row >> 6, 0);
        const uint32_t s = occ.symbol(b, row);
        if (OCC::kSymbolLoad) b = occ.load(row >> 6, s);
        n_phys += 1;
        return ix.C[s] + occ.rank(b, row, s);
    };
    // the row after m window symbols (m <= have * SPW)
    auto row_at = [&](uint32_t m) -> uint32_t {
        uint32_t row = rows[m / SPW];
        uint32_t r = m % SPW;
        if (!BYTES && r >= 4 && jv.jump4[R] != nullptr) {
#pragma unroll 1
            while (r >= 4) {
                const uint2 e = __ldg(jv.jump4[R] + row);      // valid: the window holds no delimiter
                n_phys += 1;
                row = e.x;
                r -= 4;
            }
        }
#pragma unroll 1
        while (r--) row = lf1(row);
        return row;
    };
    // fetches window word `have`; false when the window ends here (full, or a delimiter within the next SPW symbols)
    auto fetch = [&]() -> bool {
        if (closed || have == (uint32_t)kTextWords) return false;
        const uint32_t row = rows[have];
        if (!EDIT && !BYTES && jv.jshift[R] && have + 2 <= (uint32_t)kTextWords) {
            // merged LF^16 / LF^32 entries (direction 0 when the image holds them): one 16-byte lookup = 32 window symbols.  Hamming
            // instantiation only: that kernel is request bound; the edit-distance one is instruction-cache bound and lost 8 % to the
            // extra code (k = 2: 64.6 -> 70.2 ms)
            const uint4 e4 = __ldg(reinterpret_cast<const uint4*>(jv.jump[R]) + row);
            n_phys += 1;
            if (e4.x == kJumpInvalid) { closed = true; return false; }
            sw[have * 256 + tid] = R ? e4.y : rev2(e4.y);
            rows[have + 1] = e4.x;
            have += 1;
            if (e4.z != kJumpInvalid) {
                sw[have * 256 + tid] = R ? e4.w : rev2(e4.w);
                rows[have + 1] = e4.z;
                have += 1;
            }
            sw[have * 256 + tid] = 0;
            return true;
        }
        const uint2 e = BYTES ? __ldg(jv.jump4[R] + row) : __ldg(jv.jump[R] + ((size_t)row << jv.jshift[R]));
        n_phys += 1;
        if (e.x == kJumpInvalid) { closed = true; return false; }
        uint32_t w = e.y;
        if (!R) w = BYTES ? __byte_perm(w, 0, 0x0123) : rev2(w);     // direction 0 stores the nearest symbol in the high bits
        sw[have * 256 + tid] = w;
        sw[(have + 1) * 256 + tid] = 0;
        rows[have + 1] = e.x;
        have += 1;
        return true;
    };
    auto ensure = [&](uint32_t m) -> bool {
        while (m / SPW >= have)
            if (!fetch()) return false;
        return true;
    };
    auto wsym = [&](uint32_t m) -> uint32_t { return ((sw[(m / SPW) * 256 + tid] >> (B * (m % SPW))) & SM) + (BYTES ? 0u : 1u); };
    auto qsy = [&](uint32_t c) -> uint32_t { return ((sq[(c / SPW) * 256 + tid] >> (B * (c % SPW))) & SM) + (BYTES ? 0u : 1u); };
    auto wword = [&](uint32_t m) -> uint32_t { return __funnelshift_r(sw[(m / SPW) * 256 + tid], sw[(m / SPW + 1) * 256 + tid], B * (m % SPW)); };
    auto qword = [&](uint32_t c) -> uint32_t { return __funnelshift_r(sq[(c / SPW) * 256 + tid], sq[(c / SPW + 1) * 256 + tid], B * (c % SPW)); };

    // Pending hand-overs of this lane's item to the frontier kernel (served in bulk, see the R phase below), the nodes visited in
    // the current iteration (the popped node and those of its children whose own children can only continue error free) and the
    // comparisons along a diagonal queued by those visits.
    unsigned long long req[16], lc[12], mini[4];
    int nreq = 0, nlc = 0, nmini = 0;
    auto request = [&](TNode s, uint32_t kind) {
        s.kind = kind;
        req[nreq++] = tnode_pack(s);
    };
    auto push = [&](TNode s) {
        s.kind = TN_EXPAND;
        if (top < kTextStack) stk[top++] = tnode_pack(s);
        else request(s, TN_CONT);
    };
    auto queue_run = [&](TNode s, uint32_t kind) {
        s.kind = kind;
        lc[nlc++] = tnode_pack(s);
    };
    // symbols that match from (m, c), at most `limit`; status 0: stopped at a mismatch, 1: limit reached, 2: the window or the loaded
    // part of the query ends at m + result / c + result
    auto match_run = [&](uint32_t m, uint32_t c, uint32_t limit, uint32_t& status) -> uint32_t {
        uint32_t done = 0;
        status = 1;
#pragma unroll 1
        while (done < limit) {
            if (c + done >= q_limit || !ensure(m + done)) { status = 2; break; }
            uint32_t n = have * SPW - (m + done);
            n = n < SPW ? n : SPW;
            n = n < limit - done ? n : limit - done;
            n = n < q_limit - (c + done) ? n : q_limit - (c + done);
            const uint32_t x = wword(m + done) ^ qword(c + done);
            uint32_t first = SPW;
            if (BYTES) {
                uint32_t y = x | (x >> 4);
                y |= y >> 2;
                y |= y >> 1;
                y &= 0x01010101u;
                if (y) first = (uint32_t)(__ffs(y) - 1) / 8u;
            } else {
                const uint32_t y = (x | (x >> 1)) & 0x55555555u;
                if (y) first = (uint32_t)(__ffs(y) - 1) / 2u;
            }
            if (first < n) { done += first; status = 0; break; }
            done += n;
        }
        return done;
    };

    for (;;) {
        __syncwarp();
        // ---- flush the warp's staged items -------------------------------------------------------------------------------
        const bool busy = top > 0;
        const bool wants = !busy && (nreq > 0 || next_item < n_items);          // this lane needs the R / I phases to go on
        {
            const uint32_t n = stage_cnt[warp];
            const bool all_done = !__any_sync(0xFFFFFFFFu, busy || wants);
            if (n >= 32 || (all_done && n > 0)) {
                // hand-overs go to the overflow list, hits to the hit list: one counter update per kind and 32 entries
                for (uint32_t i0 = 0; i0 < n; i0 += 32) {
                    const uint32_t i = i0 + lane;
                    Item it{};
                    if (i < n) it = stage[warp][i];
                    const bool is_hit = i < n && it.meta == kHitMark;
                    // text class again (every hand-over is a single row of an unflagged query and not a leaf): not flagged `notext`, and
                    // not an error-free stretch of the generic layout (those stay in the frontier kernel, text_class())
                    const bool is_text = i < n && !is_hit && !(it.meta & 0x80u) && !(BYTES && ((it.meta >> 24) & 3u) == MODE_NOERR);
                    const bool is_item = i < n && !is_hit && !is_text;
                    const uint32_t hb = __ballot_sync(0xFFFFFFFFu, is_hit), ib = __ballot_sync(0xFFFFFFFFu, is_item), tb = __ballot_sync(0xFFFFFFFFu, is_text);
                    unsigned long long hbase = 0, ibase = 0, tbase = 0;
                    if (lane == 0) {
                        if (tb) tbase = atomicAdd(out.text_next_count, (unsigned long long)__popc(tb));
                        if (ib) ibase = atomicAdd(out.overflow_count, (unsigned long long)__popc(ib));
                        if (hb) {
                            hbase = atomicAdd(out.hit_count, (unsigned long long)__popc(hb));
                            atomicAdd(out.row_count, (unsigned long long)__popc(hb));
                        }
                    }
                    hbase = __shfl_sync(0xFFFFFFFFu, hbase, 0);
                    ibase = __shfl_sync(0xFFFFFFFFu, ibase, 0);
                    tbase = __shfl_sync(0xFFFFFFFFu, tbase, 0);
                    const uint32_t below = (1u << lane) - 1u;
                    if (is_text) {
                        const unsigned long long g = tbase + __popc(tb & below);
                        if (g < out.text_capacity) out.text_next[g] = it;
                    }
                    if (is_item) {
                        const unsigned long long g = ibase + __popc(ib & below);
                        if (g < out.overflow_capacity) out.overflow[g] = it;
                    }
                    if (is_hit) {
                        const unsigned long long g = hbase + __popc(hb & below);
                        if (g < out.hit_capacity) out.hits[g] = hit_of_item(it);
                    }
                }
                __syncwarp();
                if (lane == 0) stage_cnt[warp] = 0;
                __syncwarp();
            }
            if (all_done) break;
        }
        // ---- R / I phases: the rare, expensive steps (row computation + item packing; item fetch + query window) run when a quarter
        //      of the warp waits for them -- or nobody can go on otherwise -- so that their instructions are issued for many lanes
        const uint32_t n_wants = __popc(__ballot_sync(0xFFFFFFFFu, wants));
        const bool serve = n_wants >= 8 || (n_wants > 0 && !__any_sync(0xFFFFFFFFu, busy)) || __any_sync(0xFFFFFFFFu, nreq >= 4);
        if (serve) {
            // ---- R: hand-overs: the entry state moved to (m, c) with the node's fields
#pragma unroll 1
            for (int i = 0; __any_sync(0xFFFFFFFFu, i < nreq); ++i) {
                if (i < nreq) {
                    const TNode s = tnode_unpack(req[i]);
                    State ch = unpack_item(it0);
                    const uint32_t row = row_at(s.m);
                    if (R) ch.lb_rev = row; else ch.lb = row;
                    ch.steps += s.m;
                    if (R) ch.RInfo = s.T; else ch.LInfo = s.T;
                    // a hand-over that ends the search (the last part is over: search_next, :98-117) is a leaf: reported here (staged per
                    // warp) instead of travelling to the frontier kernel as an item.  (Measured and dropped: letting the lane continue
                    // with one of its own hand-overs -- a new direction run in the same lane -- instead of the next pass: the warps then
                    // mix the classes the host sorted them by, k = 1 / 2 edit 18.8 -> 21.9 / 67.0 -> 82.5 ms.)
                    const bool leaf = s.kind == TN_TURN ? s.part + 1 == np : (s.kind == TN_NEXT && s.part == np);
                    if (leaf) {
                        const bool ok = !EDIT || PSEUDO || ((ch.LInfo == INFO_M || ch.LInfo == INFO_I) && (ch.RInfo == INFO_M || ch.RInfo == INFO_I));
                        if (ok && sp.l[search][np - 1] <= s.e && s.e <= sp.u[search][np - 1]) {
                            HitRec h;
                            h.qidx = ch.qidx + out.qidx_base; h.lb = ch.lb; h.lb_rev = sp.zero_lb_rev ? 0 : ch.lb_rev; h.len = 1; h.steps = ch.steps; h.e = s.e;
                            stage_emit(item_of_hit(h));
                        }
                    } else {
                        if (R) ch.qposR = (ch.qposR + s.c) & 0xFFFF; else ch.qposL = (ch.qposL - s.c) & 0xFFFF;
                        ch.part = s.part; ch.pev = s.pev; ch.e = s.e;
                        ch.side = side_set(side_set(ch.side, R, 0, s.lastRank), R, 1, s.lastQRank);
                        ch.mode = s.kind == TN_TURN ? MODE_POS : (s.kind == TN_NEXT ? MODE_NEXT : (s.noerr ? MODE_NOERR : MODE_POS));
                        ch.NextPos = s.kind == TN_TURN ? 1u : 0u;
                        ch.Right = R; ch.notext = 0;
                        stage_emit(pack_item(ch));
                    }
                }
            }
            nreq = 0;
            // ---- I: next item
            if (top == 0 && next_item < n_items) {
                const Item it = items[next_item];
                next_item += stride;
                State st = unpack_item(it);
                bool ok = st.len == 1;
                if (ok && st.mode == MODE_POS && st.NextPos) {                                     // search_next_pos :119-141
                    if (st.Right) st.qposR = (st.qposR + 1) & 0xFFFF; else st.qposL = (st.qposL - 1) & 0xFFFF;
                    st.pev -= 1;
                    if (st.pev == 0) {
                        st.part += 1;
                        if (st.part != np) st.pev = sp.partition[sp.pi[st.search][st.part]];
                        st.mode = MODE_NEXT;
                    }
                }
                if (ok && st.mode == MODE_NEXT) {                                                   // search_next :98-117
                    if (st.part == np) ok = false;                                                  // a leaf: the frontier kernel reports it
                    else {
                        st.Right = (st.part == 0) || (sp.pi[st.search][st.part - 1] < sp.pi[st.search][st.part]);
                        if (sp.force_left) st.Right = 0;
                    }
                }
                if (ok) {
                    R = st.Right;
                    search = st.search;
                    rows[0] = R ? st.lb_rev : st.lb;
                    have = 0;
                    closed = false;
                    ok = fetch();
                }
                if (!ok) {
                    Item back = it;
                    back.meta |= 0x80u;                      // notext: expand this one on the index
                    stage_emit(back);
                } else {
                    const bool entry_noerr = st.mode == MODE_NOERR;
                    st.mode = MODE_POS; st.NextPos = 0; st.notext = 0;
                    it0 = pack_item(st);
                    // query symbols of this direction run in walking order
                    const uint64_t qbase = qoff[st.qidx];
                    const uint32_t qlen = (uint32_t)(qoff[st.qidx + 1] - qbase);
                    const uint32_t run = R ? qlen - st.qposR : st.qposL + 1;
                    q_limit = run < QCAP ? run : QCAP;
                    const uint32_t nw = (q_limit + SPW - 1) / SPW;
#pragma unroll 1
                    for (uint32_t k = 0; k < (uint32_t)kTextQWords + 1; ++k) {
                        uint32_t w = 0;
                        if (k < nw) {
                            if (BYTES) {
#pragma unroll 1
                                for (uint32_t j = 0; j < 4; ++j) {
                                    const long long at = R ? (long long)(qbase + st.qposR + 4 * k + j) : (long long)(qbase + st.qposL) - (long long)(4 * k + j);
                                    const uint32_t b = (at >= 0 && 4 * k + j < run) ? __ldg(qsym + at) : 0u;
                                    w |= b << (8 * j);
                                }
                            } else if (R) {
                                const uint64_t bit = 2 * (qbase + st.qposR + 16 * k);
                                const uint32_t wi = (uint32_t)(bit >> 5);
                                w = __funnelshift_r(__ldg(jv.qpk + wi), __ldg(jv.qpk + wi + 1), (uint32_t)bit & 31u);
                            } else {
                                // walking symbols 16k .. 16k+15 are the forward symbols qposL-16k-15 .. qposL-16k, reversed
                                const long long p0 = (long long)(qbase + st.qposL) - (long long)(16 * k + 15);
                                uint32_t v;
                                if (p0 >= 0) {
                                    const uint64_t bit = 2 * (uint64_t)p0;
                                    const uint32_t wi = (uint32_t)(bit >> 5);
                                    v = __funnelshift_r(__ldg(jv.qpk + wi), __ldg(jv.qpk + wi + 1), (uint32_t)bit & 31u);
                                } else {
                                    v = __ldg(jv.qpk) << (2 * (uint32_t)(-p0));      // before the first query: those fields are never read
                                }
                                w = rev2(v);
                            }
                        }
                        sq[k * 256 + tid] = w;
                    }
                    TNode root;
                    root.m = 0; root.c = 0; root.part = st.part; root.pev = st.pev; root.e = st.e;
                    root.T = R ? st.RInfo : st.LInfo;
                    root.lastRank = side_get(st.side, R, 0); root.lastQRank = side_get(st.side, R, 1);
                    root.noerr = entry_noerr ? 1u : 0u;      // an error-free stretch that became a single row
                    root.kind = TN_EXPAND;
                    stk[top++] = tnode_pack(root);
                }
            }
        }
        // ---- V: the popped node, then those of its children whose own children can only continue error free -----------------------
        nmini = 0;
        if (top > 0) mini[nmini++] = stk[--top];
#pragma unroll 1
        for (int vi = 0; __any_sync(0xFFFFFFFFu, vi < nmini); ++vi) {
            if (vi >= nmini) continue;
            const TNode s = tnode_unpack(mini[vi]);
            if (s.noerr) { queue_run(s, LC_RUN); continue; }
            if (s.c >= q_limit || !ensure(s.m)) { request(s, TN_CONT); continue; }      // the window ends here: the frontier kernel continues
            // ---- search_next_dir_single :251-365
            const uint32_t lp = sp.l[search][s.part], up = sp.u[search][s.part];
            const uint32_t sym = wsym(s.m), q = qsy(s.c);
            const bool Deletion = EDIT && (PSEUDO || (s.T != INFO_S && s.T != INFO_I));
            const bool Insertion = EDIT && (PSEUDO || (s.T != INFO_S && s.T != INFO_D));
            const bool insAllowed = (s.pev > 1 || lp <= s.e + 1) && s.e + 1 <= up;
            const bool mismatchAllowed = s.e + 1 <= up;
            const bool matchAllowed = (s.pev > 1 || lp <= s.e) && s.e <= up &&
                                      (PSEUDO || ((s.T != INFO_I || q != s.lastQRank) && (s.T != INFO_D || q != s.lastRank)));
            const bool eq = sym == q;
            n_ext += 1;
            if (eq && matchAllowed && !mismatchAllowed) {
                queue_run(s, LC_RUN);                                    // same node again inside the error-free loop (:311-315)
                continue;
            }
            // the three children in one shape: 0 = along the diagonal (match / substitution), 1 = deletion, 2 = insertion
            const uint32_t exists = ((eq ? (matchAllowed && mismatchAllowed) : (mismatchAllowed && insAllowed)) ? 1u : 0u) |
                                    ((Deletion && mismatchAllowed) ? 2u : 0u) | ((Insertion && insAllowed) ? 4u : 0u);
#pragma unroll 1
            for (uint32_t slot = 0; slot < 3; ++slot) {
                if (!((exists >> slot) & 1)) continue;
                TNode ch = s;
                const bool adv = slot != 1;                              // the child consumes the query symbol (search_next_pos)
                if (slot != 2) { ch.m += 1; ch.lastRank = sym; }
                if (slot != 1) ch.lastQRank = q;
                if (slot != 0 || !eq) ch.e += 1;
                ch.T = slot == 0 ? (eq ? INFO_M : INFO_S) : (slot == 1 ? INFO_D : INFO_I);
                if (adv) {
                    if (ch.pev == 1) {                                   // the advance ends the part
                        const uint32_t next = ch.part + 1;
                        if (next == np || sp.force_left || dir_of(next) != R) {
                            request(ch, TN_TURN);                        // the search ends or turns around: the child as it is, advance pending
                            continue;
                        }
                        ch.part = next;
                        ch.pev = sp.partition[sp.pi[search][next]];
                    } else {
                        ch.pev -= 1;
                    }
                    ch.c += 1;
                }
                const uint32_t cup = sp.u[search][ch.part];
                if (ch.e >= cup) {
                    queue_run(ch, LC_VISIT);                             // no error left: its own visit, then error free
                } else if (!PSEUDO && slot == 0 && eq && (EDIT ? ch.e + 1 == cup : true) && ch.pev > 1 && ch.part == s.part) {
                    queue_run(ch, LC_SKIP);                              // the matching stretch (edit distance: at the last error level) is skipped
                } else if (EDIT && !PSEUDO && !BYTES && slot == 0 && eq && ch.e + 2 == cup && ch.pev >= 4 && ch.part == s.part) {
                    queue_run(ch, LC_BULK2);                             // two errors left: the stretch is evaluated 16 positions at a time
                } else if (vi == 0 && !(slot == 0 && eq) && ch.e + 1 == cup && nmini < 4) {
                    ch.kind = TN_EXPAND;
                    mini[nmini++] = tnode_pack(ch);                      // visited in this iteration
                } else {
                    push(ch);
                }
            }
        }
        // ---- L: comparisons along a diagonal -------------------------------------------------------------------------------------------
#pragma unroll 1
        for (int li = 0; __any_sync(0xFFFFFFFFu, li < nlc); ++li) {
            if (li >= nlc) continue;
            TNode s = tnode_unpack(lc[li]);
            uint32_t status;
            if (s.kind == LC_SKIP) {
                // Edit distance, last error level, inside the part, after a match: while the text keeps matching, every node that is not
                // the part's last has the same three visits -- itself, its deletion child (dies: it would have to match the symbol it
                // just deleted, :275) and its insertion child (dies: it would have to match the symbol it just inserted).  Hamming
                // distance: a matching node has its match child only, at every error level.
                const uint32_t j = match_run(s.m, s.c, s.pev - 1, status);
                if (j) {
                    n_ext += (EDIT ? 3 : 1) * j;
                    s.m += j; s.c += j; s.pev -= j;
                    s.lastRank = s.lastQRank = qsy(s.c - 1);
                }
                push(s);
                continue;
            }
            if constexpr (EDIT && !PSEUDO && !BYTES) {
                if (s.kind == LC_BULK2) {
                    // the matching stretch of a path with two errors left, sixteen positions per evaluation (bulk2_eval above); positions
                    // that are not decided there get their own visit here and their two children on the stack
                    const uint32_t m0 = s.m, c0 = s.c, pev0 = s.pev;
                    const uint32_t last = pev0 - 1 < 31u ? pev0 - 1 : 31u;         // positions c0 .. c0 + last matter
                    // the query symbols the masks read lie inside the loaded part of the query (those beyond the part do not matter)
                    if (c0 + 18 <= QCAP && c0 + (pev0 < last + 3 ? pev0 : last + 3) <= q_limit && ensure(m0 + last + 2)) {
                        uint32_t nb = 0;
                        unsigned long long slow = 0;
                        const uint32_t total = bulk2_eval(sw, sq, tid, have * SPW, m0, c0, pev0, nb, slow);
                        if (nb) {
                            n_ext += total;
                            while (slow) {
                                const uint32_t i = (uint32_t)(__ffsll((long long)slow) - 1) / 2u;
                                slow &= slow - 1;
                                const uint32_t qc = qsy(c0 + i);
                                TNode d1 = s;                                      // deletion child of the node at (m0 + i, c0 + i)
                                d1.m = m0 + i + 1; d1.c = c0 + i; d1.pev = pev0 - i; d1.e = s.e + 1; d1.T = INFO_D; d1.lastRank = qc;
                                d1.lastQRank = i ? qsy(c0 + i - 1) : s.lastQRank;
                                push(d1);
                                TNode i1 = s;                                      // insertion child: consumes q[c0 + i]
                                i1.m = m0 + i; i1.c = c0 + i + 1; i1.pev = pev0 - i - 1; i1.e = s.e + 1; i1.T = INFO_I; i1.lastQRank = qc;
                                i1.lastRank = i ? qsy(c0 + i - 1) : s.lastRank;
                                push(i1);
                            }
                            s.m += nb; s.c += nb; s.pev -= nb;
                            s.lastRank = s.lastQRank = qsy(s.c - 1);
                        }
                    }
                    push(s);                                                       // the path goes on with the node behind the block (or unchanged)
                    continue;
                }
            }
            if (s.kind == LC_VISIT) {
                // the node's own visit (search_next_dir_single with no error left): it continues iff its symbol matches
                if (s.c >= q_limit || !ensure(s.m)) { request(s, TN_CONT); continue; }
                const uint32_t lp = sp.l[search][s.part], up = sp.u[search][s.part];
                const uint32_t q = qsy(s.c);
                n_ext += 1;
                const bool matchAllowed = (s.pev > 1 || lp <= s.e) && s.e <= up &&
                                          (PSEUDO || ((s.T != INFO_I || q != s.lastQRank) && (s.T != INFO_D || q != s.lastRank)));
                if (wsym(s.m) != q || !matchAllowed) continue;
            }
            // search_next_dir_no_errors (:225-250): the rest of the part must match
            const uint32_t j = match_run(s.m, s.c, s.pev, status);
            if (status == 0) { n_ext += j + 1; continue; }               // the path dies at that symbol
            n_ext += j;
            s.m += j; s.c += j; s.pev -= j;
            if (status == 2) { s.noerr = 1; request(s, TN_CONT); continue; }
            {                                                            // :241-249
                const uint32_t lastq = qsy(s.c - 1);
                const uint32_t next = s.part + 1;
                s.part = next;
                s.pev = (next != np) ? sp.partition[sp.pi[search][next]] : 0u;
                s.T = INFO_M; s.lastRank = lastq; s.lastQRank = lastq; s.noerr = 0;
                if (next == np || sp.force_left || dir_of(next) != R) request(s, TN_NEXT);
                else push(s);
            }
        }
        nlc = 0;
    }

    // ---- statistics: every visit / compared symbol is one extension and one occ lookup of the reference's walk -------------------
    for (int o = 16; o > 0; o >>= 1) {
        n_ext += __shfl_xor_sync(0xFFFFFFFFu, n_ext, o);
        n_phys += __shfl_xor_sync(0xFFFFFFFFu, n_phys, o);
    }
    if (lane == 0) {
        atomicAdd(out.counters + CTR_EXTENSIONS, (unsigned long long)n_ext);
        atomicAdd(out.counters + CTR_OCC_LOOKUPS, (unsigned long long)n_ext);
        atomicAdd(out.counters + CTR_LINE_REQUESTS, (unsigned long long)n_phys);
    }
}

}  // namespace fmb
