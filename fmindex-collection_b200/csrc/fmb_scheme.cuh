// fmb_scheme.cuh -- K3: k-error search with search schemes (Hamming / Edit) and backtracking on sm_100a.
//
// Semantics = search_ng26 of the reference (search/SearchNg26.h:18-366): the node state machine
// search_next / search_next_pos / search_next_dir / search_next_dir_no_errors / search_next_dir_single is
// reproduced exactly (same pruning, same children), only the traversal order differs: the reference recurses
// depth first per query, here every WARP owns a shared-memory stack of pending states ("items") of many
// queries.  Per iteration the warp pops up to 32 items, every lane expands ONE node (one or two occ-block
// fetches), the children are compacted with a warp prefix sum and pushed back.  Lanes therefore always work
// on different, independent (query, search, position, interval) items -- the breadth-first frontier of the
// north star, staged in shared memory, with LIFO order to keep it bounded.  New roots (query x search pairs)
// are pulled from a global counter whenever fewer than 32 items are pending; children that do not fit the
// stack are spilled to a global overflow list that the host feeds into the next launch.
//
// Because no hit limit (`n`) is applied, the set of reported (cursor, e) pairs does not depend on the
// traversal order (SURVEY.md §0 fact 5, §7 "hard parts").
#pragma once
#include "fmb_device.cuh"
#include "fmb_host.hpp"

namespace fmb {

constexpr int kMaxSearches = 16;
constexpr int kMaxParts = 16;

struct SchemeParams {
    uint32_t n_searches, n_parts;
    uint32_t edit;            // 1 = edit distance, 0 = Hamming
    uint32_t force_left;      // backtracking mode: a single part searched right-to-left (search/Backtracking.h)
    uint32_t zero_lb_rev;     // unidirectional index: report lb_rev = 0
    uint8_t pi[kMaxSearches][kMaxParts];
    uint8_t l[kMaxSearches][kMaxParts];
    uint8_t u[kMaxSearches][kMaxParts];
    uint16_t partition[kMaxParts];
    uint16_t start[kMaxSearches];      // sum of partition[0 .. pi[s][0])          (SearchNg26.h:65-68)
    // ordered mode (hit limit n, SearchNg26.h:408-423): layout of the discovery-order key, see order_key_edge
    uint32_t key_slots, key_bits, key_maxd, key_ords;
};

enum : uint32_t { INFO_M = 0, INFO_S = 1, INFO_D = 2, INFO_I = 3 };
enum : uint32_t { MODE_POS = 0, MODE_NEXT = 1, MODE_NOERR = 2 };

// 32-byte frontier item = State of SearchNg26.h:41-52 + (qidx, search)
struct alignas(16) Item {
    uint32_t lb, lb_rev, len, qidx;
    uint32_t qpos;       // queryPosL | queryPosR << 16  (16-bit wrap-around, cf. the note at SearchNg26.h:69-71)
    uint32_t pev_steps;  // partitionEntryValue | steps << 16
    uint32_t meta;       // e (7 bits) | notext << 7 | part << 8 | search << 16 | mode << 24 | LInfo << 26 | RInfo << 28 | Right << 30 | NextPos << 31
    uint32_t side;       // lastRank[L] | lastQRank[L] << 8 | lastRank[R] << 16 | lastQRank[R] << 24
};
static_assert(sizeof(Item) == 32, "item is two 16-byte words");

struct State {
    uint32_t lb, lb_rev, len, qidx;
    uint32_t qposL, qposR, pev, steps;
    uint32_t e, part, search, mode, LInfo, RInfo, Right, NextPos;
    uint32_t notext;     // the text kernel handed this single-row item back (no usable text window at its row): expand it on the index
    uint32_t side;
    unsigned long long key;   // ordered mode only (not part of Item: kept in a parallel stack)
};

__device__ __forceinline__ Item pack_item(const State& s) {
    Item it;
    it.lb = s.lb; it.lb_rev = s.lb_rev; it.len = s.len; it.qidx = s.qidx;
    it.qpos = (s.qposL & 0xFFFF) | (s.qposR << 16);
    it.pev_steps = (s.pev & 0xFFFF) | (s.steps << 16);
    it.meta = s.e | (s.notext << 7) | (s.part << 8) | (s.search << 16) | (s.mode << 24) | (s.LInfo << 26) | (s.RInfo << 28) | (s.Right << 30) | (s.NextPos << 31);
    it.side = s.side;
    return it;
}
__device__ __forceinline__ State unpack_item(const Item& it) {
    State s;
    s.lb = it.lb; s.lb_rev = it.lb_rev; s.len = it.len; s.qidx = it.qidx;
    s.qposL = it.qpos & 0xFFFF; s.qposR = it.qpos >> 16;
    s.pev = it.pev_steps & 0xFFFF; s.steps = it.pev_steps >> 16;
    s.e = it.meta & 0x7F; s.notext = (it.meta >> 7) & 1; s.part = (it.meta >> 8) & 0xFF; s.search = (it.meta >> 16) & 0xFF;
    s.mode = (it.meta >> 24) & 3; s.LInfo = (it.meta >> 26) & 3; s.RInfo = (it.meta >> 28) & 3;
    s.Right = (it.meta >> 30) & 1; s.NextPos = it.meta >> 31;
    s.side = it.side;
    return s;
}
__device__ __forceinline__ uint32_t side_get(uint32_t side, uint32_t right, uint32_t which /*0 lastRank, 1 lastQRank*/) {
    return (side >> (right * 16 + which * 8)) & 0xFF;
}
__device__ __forceinline__ uint32_t side_set(uint32_t side, uint32_t right, uint32_t which, uint32_t v) {
    uint32_t sh = right * 16 + which * 8;
    return (side & ~(0xFFu << sh)) | (v << sh);
}

// Discovery-order key (ordered mode).  With a hit limit the reference stops a query after its first n rows IN THE ORDER ITS
// DEPTH-FIRST SEARCH FINDS THEM (search_n_impl, SearchNg26.h:408-423).  The kernel enumerates the tree in its own order, so every
// item carries a sparse key from which that order is recovered afterwards by sorting.  Two paths of one search split at one node
// and their order is the order in which that node visits the two children:
//   search_next_dir        (:170-218)  match, then for every symbol c: deletion(c), substitution(c), then insertion
//   search_next_dir_single (:286-363)  insertion, then match / deletion  or  substitution / deletion
// so a path is identified by its error edges.  Slot e of the key (e = errors before the edge; top byte = search number, slots
// follow from the high bits down) holds a code for the error edge leaving a node of depth d = steps + e (strictly increasing
// along a path):
//   insertion at a single-row node (visited before the match child)     code = d
//   no further error edge                                                 code = MID = key_maxd
//   any other error edge (visited after the match child)                  code = MID + 1 + (key_maxd - 1 - d) * key_ords + ord
// ord = 0 substitution / 1 deletion at a single-row node; 2c deletion(c) / 2c + 1 substitution(c) / 2 sigma + 1 insertion at a
// wide node.  Mismatches absorbed by a multi-symbol jump (Hamming) lie on single-row nodes with exactly one child and need no
// entry.  Unsigned comparison of two keys = order of discovery (the tests check the definition against the report order of
// the reference's depth-first search).
__device__ __forceinline__ unsigned long long order_key_edge(const SchemeParams& sp, unsigned long long key, uint32_t steps, uint32_t e,
                                                             bool before, uint32_t ord) {
    const uint32_t d = steps + e;
    const unsigned long long code = before ? (unsigned long long)d
                                           : (unsigned long long)sp.key_maxd + 1 + (unsigned long long)(sp.key_maxd - 1 - d) * sp.key_ords + ord;
    const uint32_t sh = 56 - (e + 1) * sp.key_bits;
    const unsigned long long mask = ((1ull << sp.key_bits) - 1) << sh;
    return (key & ~mask) | (code << sh);
}
__device__ __forceinline__ unsigned long long order_key_root(const SchemeParams& sp, uint32_t search) {
    unsigned long long key = (unsigned long long)search << 56;
    for (uint32_t i = 0; i < sp.key_slots; ++i) key |= (unsigned long long)sp.key_maxd << (56 - (i + 1) * sp.key_bits);
    return key;
}

// slots of the counter block of a search call: the statistics (SchemeOut::counters points at CTR_EXTENSIONS) and the list counters
enum : uint32_t {
    CTR_EXTENSIONS = 0, CTR_OCC_LOOKUPS = 1, CTR_LINE_REQUESTS = 2, CTR_PEAK = 3,
    CTR_HITS = 4, CTR_OVERFLOW = 5, CTR_ROOTS = 6, CTR_TEXT_A = 7, CTR_ROWS = 8, CTR_TEXT_B = 9,
    CTR_SLOTS = 10
};

struct SchemeOut {
    HitRec* hits;
    unsigned long long* hit_count;     // total hits found (may exceed capacity)
    unsigned long long* row_count;     // sum of the interval lengths of all hits (what locate will have to produce)
    uint64_t hit_capacity;
    Item* overflow;
    unsigned long long* overflow_count;
    uint64_t overflow_capacity;
    unsigned long long* counters;      // [CTR_EXTENSIONS], [CTR_OCC_LOOKUPS], [CTR_LINE_REQUESTS], [CTR_PEAK] peak items per warp
    unsigned long long* root_counter;
    uint32_t qidx_base;                // added to the reported qidx (chunked query batches)
    uint64_t root_base;                // first root (query x search pair) of this launch's slab
    // text list: single-row items of edit-distance searches, handed to scheme_text_kernel (null: not used)
    Item* text;
    unsigned long long* text_count;
    uint64_t text_capacity;
    // text kernel only: the text list of the NEXT pass -- its text-class hand-overs (a new direction run, a new window) go there
    // directly instead of through the overflow list and a routing launch of the frontier kernel
    Item* text_next;
    unsigned long long* text_next_count;
    // ordered mode: keys of the hits / the spilled items / the items fed in
    unsigned long long* hit_keys;
    unsigned long long* overflow_keys;
    const unsigned long long* in_keys;
    // hit limit n <= kMaxPruneN: best_keys[q * prune_n + i] = the (i + 1)-th smallest discovery-order key among the rows of query q found
    // so far (all ones: none; a hit of len rows counts min(len, n) times); subtrees whose smallest possible key is larger than the n-th
    // cannot hold one of the first n rows and are dropped.  n_queries > 0 additionally orders the roots search by search (all queries'
    // search 0, then search 1, ...), so that the later searches of a query start after its earlier hits exist.
    unsigned long long* best_keys;
    uint64_t n_queries;
    uint32_t prune_n;
};
constexpr uint32_t kMaxPruneN = 8;

// the key no later row of query q can exceed and still be among its first n rows
__device__ __forceinline__ unsigned long long prune_bound(const SchemeOut& out, uint32_t qidx) {
    return __ldcg(out.best_keys + (size_t)qidx * out.prune_n + (out.prune_n - 1));
}
// A row with key `key` was found: bubble it into the query's n smallest.  Every step is one atomicMin whose displaced (larger) value is
// carried to the next slot, so the slots only ever decrease and the multiset {slots, values in flight} is preserved: whenever slot n-1
// holds x, slots 0 .. n-2 hold -- now and later -- other rows with keys <= x, i.e. x is a valid bound at any moment, not only at rest.
__device__ __forceinline__ void prune_insert(const SchemeOut& out, uint32_t qidx, unsigned long long key, uint32_t copies) {
    unsigned long long* slots = out.best_keys + (size_t)qidx * out.prune_n;
    copies = copies < out.prune_n ? copies : out.prune_n;
    for (uint32_t c = 0; c < copies; ++c) {
        unsigned long long k = key;
        for (uint32_t i = c; i < out.prune_n && k != ~0ull; ++i) {
            const unsigned long long old = atomicMin(slots + i, k);
            k = old > k ? old : k;
        }
    }
}

// smallest discovery-order key a descendant of a node (e errors so far, depth = steps + e) can end with: the slots of errors still to
// come hold at least the code of an insertion at the node itself (the only codes below "no further error"; edit distance only)
template <bool EDIT>
__device__ __forceinline__ unsigned long long order_key_lower_bound(const SchemeParams& sp, unsigned long long key, uint32_t steps, uint32_t e) {
    if (!EDIT || e >= sp.key_slots) return key;
    const uint32_t sh = 56 - (e + 1) * sp.key_bits;
    const unsigned long long below = (sh + sp.key_bits >= 64) ? ~0ull : ((1ull << (sh + sp.key_bits)) - 1);
    return (key & ~below) | ((unsigned long long)(steps + e) << sh);
}

// one cursor extension by `symb` in direction `right` from two loaded blocks (DNA: blocks are symbol independent)
template <class OCC>
__device__ __forceinline__ void child_cursor(const IndexView<OCC>& ix, const OCC& occ, uint32_t b0, uint32_t b1,
                                             typename OCC::Block& blk0, typename OCC::Block& blk1, row_t lo, row_t hi,
                                             uint32_t symb, bool single, uint32_t& same, uint32_t& dother, uint32_t& clen) {
    if (single) {
        // interval of one row whose BWT symbol is `symb` (callers guarantee it): rank(lo+1) = rank(lo) + 1 and no
        // smaller symbol lies inside, so the second block -- lo + 1 may start the next one -- is never needed
        if (OCC::kSymbolLoad) blk0 = occ.load(b0, symb);
        same = ix.C[symb] + occ.rank(blk0, lo, symb);
        dother = 0;
        clen = 1;
        return;
    }
    if (OCC::kSymbolLoad) {
        blk0 = occ.load(b0, symb);
        blk1 = (b1 == b0) ? blk0 : occ.load(b1, symb);
    }
    uint32_t r0, p0, r1, p1;
    occ.rank_pr(blk0, lo, symb, r0, p0);
    occ.rank_pr(blk1, hi, symb, r1, p1);
    same = ix.C[symb] + r0;
    dother = p1 - p0;
    clen = r1 - r0;
}

// LF^16 jump tables of both directions + the 2-bit packed queries (DNA layout only; all pointers may be null)
struct JumpView {
    const uint2* jump[2];         // [0]: farthest symbol in the low bits, [1]: nearest symbol in the low bits (= query order)
    const uint2* jump4[2];        // LF^4 tables, same orientation, four symbols in the low 8 bits
    uint32_t jshift[2];           // 1: jump[d] holds 16-byte merged LF^16 / LF^32 entries, the LF^16 part first (row r at jump[d] + 2 r)
    const uint32_t* qpk;          // packed query symbols
    const uint8_t* qflags;        // 1 = query not packable
    // bidirectional k-mer table: entry (2-bit packed k-mer, first symbol in the low bits) = {lb, lbRev, len, work} of the
    // pattern after bikmer_k extendRight steps from the whole index; work = extensions << 16 | occ lookups the reference
    // spends on those steps (fewer than k extensions when the pattern does not occur).  Serves roots whose first part
    // is error free: the wide-interval phase of every search becomes one lookup.
    const uint4* bikmer;
    uint32_t bikmer_k;
    uint32_t bikmer_base;         // generic layout: the k-mer index is the base-`bikmer_base` number of (symbol - first_symb); 0: 2-bit packed key
};

// ---------------------------------------------------------------------------------------------------------------------
// Window simulation of a single-row subtree (edit distance).
// On a single-row interval the search walks the text: the row after t consumed text symbols is LF^t(row) and the symbols it
// meets are the entries of jump[row] (16 of them in one 8-byte lookup).  So the fate of an error child can be decided here,
// without touching the index: the subtree is expanded with exactly the rules of search_next_dir_single /
// search_next_dir_no_errors / search_next_pos (SearchNg26.h:119-141, 225-365) on the window symbols.  If every path dies
// inside the window the child is never created and only its extensions are counted; if some path reaches the window end, a
// part that changes direction, or the end of the search, the simulation gives up and the child is created as usual.
// ---------------------------------------------------------------------------------------------------------------------
// a path still alive after SIM_DEPTH window symbols counts as a survivor (measured: 8 is as good as the full 16)
#ifndef SIM_DEPTH
#define SIM_DEPTH 8
#endif
#ifndef SIM_BUDGET
#define SIM_BUDGET 96
#endif
struct SimState {          // one pending node, "ready to expand" (the NextPos advance already applied)
    uint32_t m;            // text symbols consumed inside the window: the node looks at w[m]
    uint32_t c;            // query symbols consumed since the window started
    uint32_t part, pev, e;
    uint32_t T;            // info of the walking side (INFO_*)
    uint32_t lastRank, lastQRank;
    uint32_t noerr;        // inside the error-free loop
};
__device__ __forceinline__ unsigned long long sim_pack(const SimState& s) {
    // m:5 c:8 part:4 pev:16 e:4 T:2 lastRank:8 lastQRank:8 noerr:1  (symbols up to 255: the generic layout has sigma <= 32)
    return (unsigned long long)s.m | ((unsigned long long)s.c << 5) | ((unsigned long long)s.part << 13) | ((unsigned long long)s.pev << 17) |
           ((unsigned long long)s.e << 33) | ((unsigned long long)s.T << 37) | ((unsigned long long)s.lastRank << 39) |
           ((unsigned long long)s.lastQRank << 47) | ((unsigned long long)s.noerr << 55);
}
__device__ __forceinline__ SimState sim_unpack(unsigned long long v) {
    SimState s;
    s.m = v & 31; s.c = (v >> 5) & 255; s.part = (v >> 13) & 15; s.pev = (v >> 17) & 0xFFFF; s.e = (v >> 33) & 15;
    s.T = (v >> 37) & 3; s.lastRank = (v >> 39) & 255; s.lastQRank = (v >> 47) & 255; s.noerr = (v >> 55) & 1;
    return s;
}

// BYTES: the window holds 4 symbols of 8 bits (generic layout, LF^4 table) instead of 16 codes of 2 bits (symbol - 1)
// PSEUDO: edit distance without the redundancy filter (search_pseudo's search_distance, search/SearchPseudo.h:100-165): deletions and
// insertions are allowed after every kind of step and a match may follow them
template <bool EDIT, bool BYTES, bool PSEUDO>
__device__ bool sim_subtree_dies(const SchemeParams& sp, uint32_t search, uint32_t R, uint32_t window /*w[0] in the low bits*/,
                                 const uint8_t* __restrict__ qptr /*query symbol of c = 0*/, const SimState& root, uint32_t& ext) {
    constexpr int kStack = 12;
    unsigned long long stack[kStack];
    int top = 0;
    stack[top++] = sim_pack(root);
    uint32_t count = 0;
    const uint32_t np = sp.n_parts;
    const int dirstep = R ? 1 : -1;
    int budget = SIM_BUDGET;                           // node visits; beyond that the child is simply created
    while (top > 0) {
        SimState s = sim_unpack(stack[--top]);
        if (--budget < 0) return false;
        // ---- the NextPos advance of a child: returns false when the path leaves what the window can decide
        auto advance = [&](SimState& ch) -> bool {
            ch.c += 1;
            ch.pev -= 1;
            if (ch.pev == 0) {
                ch.part += 1;
                if (ch.part == np) return false;                                                     // leaf: may report
                const uint32_t nr = (sp.pi[search][ch.part - 1] < sp.pi[search][ch.part]) ? 1u : 0u;
                if (sp.force_left || nr != R) return false;                                          // the walk turns around
                ch.pev = sp.partition[sp.pi[search][ch.part]];
            }
            return true;
        };
        if (s.m >= (BYTES ? 4u : (uint32_t)SIM_DEPTH)) return false;                                 // survives the window
        const uint32_t sym = BYTES ? ((window >> (8 * s.m)) & 0xFFu) : ((window >> (2 * s.m)) & 3u) + 1;
        const uint32_t q = qptr[dirstep * (int)s.c];
        const uint32_t lp = sp.l[search][s.part], up = sp.u[search][s.part];
        if (s.noerr) {                                                                               // search_next_dir_no_errors :225-250
            count += 1;
            if (sym != q) continue;
            SimState ch = s;
            ch.m += 1;
            ch.lastRank = q; ch.lastQRank = q;     // only read after the loop ends (set there by the reference)
            ch.c += 1; ch.pev -= 1;
            if (ch.pev == 0) {
                ch.T = INFO_M;
                ch.noerr = 0;
                ch.part += 1;
                if (ch.part == np) return false;
                const uint32_t nr = (sp.pi[search][ch.part - 1] < sp.pi[search][ch.part]) ? 1u : 0u;
                if (sp.force_left || nr != R) return false;
                ch.pev = sp.partition[sp.pi[search][ch.part]];
            } else {
                // lastRank / lastQRank / T stay those of the loop's entry until the part ends (:241-249)
                ch.lastRank = s.lastRank; ch.lastQRank = s.lastQRank;
            }
            if (top >= kStack) return false;
            stack[top++] = sim_pack(ch);
            continue;
        }
        // ---- search_next_dir_single :251-365
        const bool Deletion = EDIT && (PSEUDO || (s.T != INFO_S && s.T != INFO_I));
        const bool Insertion = EDIT && (PSEUDO || (s.T != INFO_S && s.T != INFO_D));
        const bool insAllowed = (s.pev > 1 || lp <= s.e + 1) && s.e + 1 <= up;
        const bool mismatchAllowed = s.e + 1 <= up;
        const bool matchAllowed = (s.pev > 1 || lp <= s.e) && s.e <= up && (PSEUDO || ((s.T != INFO_I || q != s.lastQRank) && (s.T != INFO_D || q != s.lastRank)));
        count += 1;
        if (top + 3 > kStack) return false;
        if (sym == q) {
            if (matchAllowed) {
                if (!mismatchAllowed) {
                    SimState ch = s;                   // same node again inside the error-free loop (:311-315)
                    ch.noerr = 1;
                    stack[top++] = sim_pack(ch);
                } else {
                    SimState ch = s;
                    ch.m += 1; ch.lastRank = q; ch.lastQRank = q; ch.T = INFO_M;
                    if (!advance(ch)) return false;
                    stack[top++] = sim_pack(ch);
                }
            }
            if (Deletion && mismatchAllowed) {
                SimState ch = s;
                ch.m += 1; ch.e += 1; ch.lastRank = sym; ch.T = INFO_D;
                stack[top++] = sim_pack(ch);
            }
        } else if (mismatchAllowed) {
            if (insAllowed) {                          // substitution
                SimState ch = s;
                ch.m += 1; ch.e += 1; ch.lastRank = sym; ch.lastQRank = q; ch.T = INFO_S;
                if (!advance(ch)) return false;
                stack[top++] = sim_pack(ch);
            }
            if (Deletion) {
                SimState ch = s;
                ch.m += 1; ch.e += 1; ch.lastRank = sym; ch.T = INFO_D;
                stack[top++] = sim_pack(ch);
            }
        }
        if (Insertion && insAllowed) {
            SimState ch = s;
            ch.e += 1; ch.lastQRank = q; ch.T = INFO_I;
            if (!advance(ch)) return false;
            stack[top++] = sim_pack(ch);
        }
    }
    ext = count;
    return true;
}

// children of one expanded node are described by a bit mask and re-derived when they are written:
//   bit 0 match / error-free continuation, bit 1 insertion, bit 2 sixteen-symbol jump,
//   bits 8+c deletion(c), bits 36+c substitution(c)
constexpr unsigned long long CH_MATCH = 1ull, CH_INS = 2ull, CH_JUMP = 4ull, CH_SELF = 8ull;    // CH_SELF: the node itself goes back (to the text list)
constexpr uint32_t kDelBit = 8, kSubBit = 36;
// the two symbol ranges of the mask must not overlap nor leave the 64 bits: k-error searches are refused above this alphabet size
constexpr uint32_t kMaxSchemeSigma = 28;
static_assert(kDelBit + kMaxSchemeSigma <= kSubBit && kSubBit + kMaxSchemeSigma <= 64, "child mask layout");
// the window simulation packs the error count of a state into 4 bits (sim_pack)
constexpr uint32_t kMaxSchemeErrors = 15;
constexpr int kFastForward = 12;
#ifndef FMB_SCHEME_MINB
#define FMB_SCHEME_MINB 4          // 4 blocks of 256 threads per SM -> 64 registers (a few spills beat the lower occupancy of 80)
#endif   // consecutive single-child expansions a lane may chain in registers per pop

// Text class: a single-row item that is not a leaf.  Its whole subtree in the current direction is decided by the text that follows
// the row, so the frontier kernel does not expand it: it hands it to scheme_text_kernel through the global text list.  Leaves (they
// only report) and items the text kernel handed back (notext: no usable window at that row) stay here.
__device__ __forceinline__ bool text_class(const State& c, uint32_t np, const uint8_t* __restrict__ qflags, bool noerr_too) {
    if (c.len != 1 || c.notext) return false;
    // error-free stretches: the text kernel compares 16 symbols per window lookup where the 2-bit layout has LF^16 entries; with the
    // byte-symbol LF^4 entries of the generic layout a window lookup covers what a jump of this kernel covers, so they stay here
    if (c.mode == MODE_NOERR && !noerr_too) return false;
    if (c.mode == MODE_NEXT ? (c.part == np) : (c.NextPos && c.pev == 1 && c.part + 1 == np)) return false;
    if (qflags != nullptr && qflags[c.qidx]) return false;
    return true;
}

template <class OCC, bool EDIT, bool ORDERED, bool PSEUDO>
__global__ void __launch_bounds__(256, FMB_SCHEME_MINB) scheme_search_kernel(const __grid_constant__ IndexView<OCC> ix, const __grid_constant__ SchemeParams sp,
                                                            const uint8_t* __restrict__ qsym, const uint64_t* __restrict__ qoff,
                                                            const __grid_constant__ JumpView jv, uint64_t n_roots,
                                                            const Item* __restrict__ in_items, uint64_t n_in,
                                                            const __grid_constant__ SchemeOut out, uint32_t cap) {
    extern __shared__ uint4 smem_raw[];
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = threadIdx.x >> 5;
    Item* stack = reinterpret_cast<Item*>(smem_raw) + (size_t)warp * cap;
    // ordered mode: the keys of the stacked items, behind the item stacks of all warps
    unsigned long long* kstack = reinterpret_cast<unsigned long long*>(reinterpret_cast<Item*>(smem_raw) + (size_t)(blockDim.x >> 5) * cap) + (size_t)warp * cap;
    const uint64_t total_roots = n_roots + n_in;
    // the warp's stack has two ends: pending items grow from stack[0] upwards (top of them), text-class items are staged from
    // stack[cap - 1] downwards (ttop of them) and flushed to the global text list 32 at a time
    constexpr bool kText = !ORDERED;                  // instantiations that can hand items to the text kernel
    const bool text_on = kText && out.text != nullptr;
    const uint8_t* text_qflags = OCC::kSymbolLoad ? nullptr : jv.qflags;
    uint32_t top = 0, ttop = 0;
    auto flush_text = [&](uint32_t count) {           // the `count` most recently staged items (warp uniform, count <= 32)
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(out.text_count, (unsigned long long)count);
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        __syncwarp();
        if (lane < count && base + lane < out.text_capacity) out.text[base + lane] = stack[cap - 1 - (ttop - count + lane)];
        ttop -= count;
        __syncwarp();
    };
    uint32_t n_ext = 0, n_look = 0, n_phys = 0, peak = 0;
    bool more_roots = true;
    const uint32_t np = sp.n_parts;
    const uint32_t first_symb = ix.first_symb;   // FirstSymb (fmindex/BiFMIndex.h:26): 1 for delimited indices, 0 for NoDelim
    // a warp keeps fast-forwarding while at least ff_min of its lanes have a single child; edit distance branches
    // at almost every node, so it only pays there when most of the warp is inside error-free stretches
    constexpr uint32_t ff_min = EDIT ? 16u : 8u;

    for (;;) {
        // ---- refill: pull roots while fewer than 32 items are pending -------------------------------------
        if (top < 32 && more_roots && top + ttop + 32 <= cap) {
            uint32_t want = 32 - top;
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(out.root_counter, (unsigned long long)want);
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            if (base >= total_roots) {
                more_roots = false;
            } else {
                uint64_t avail = total_roots - base;
                uint32_t got = avail < want ? (uint32_t)avail : want;
                if (got < want) more_roots = false;
                bool to_text = false;
                Item it;
                unsigned long long rkey = 0;
                if (lane < got) {
                    uint64_t r = base + lane;
                    if (r < n_in) {
                        it = in_items[r];
                        if constexpr (ORDERED) rkey = out.in_keys[r];
                        // items that come back from the text kernel (or were spilled) are routed by class
                        if (text_on) to_text = text_class(unpack_item(it), np, text_qflags, !OCC::kSymbolLoad);
                    } else {
                        r = r - n_in + out.root_base;
                        uint32_t s = (uint32_t)(r % sp.n_searches);
                        State st;
                        st.qidx = (uint32_t)(r / sp.n_searches);
                        if (ORDERED && out.n_queries) {                                        // search-major root order
                            s = (uint32_t)(r / out.n_queries);
                            st.qidx = (uint32_t)(r % out.n_queries);
                        }
                        st.lb = 0; st.lb_rev = 0; st.len = ix.n; st.steps = 0;                 // BiFMIndexCursor.h:28-30
                        st.qposR = sp.start[s];
                        st.qposL = (sp.start[s] - 1) & 0xFFFF;                                 // SearchNg26.h:69-72
                        st.pev = sp.partition[sp.pi[s][0]];
                        st.e = 0; st.part = 0; st.search = s; st.mode = MODE_NEXT;
                        st.LInfo = INFO_M; st.RInfo = INFO_M; st.Right = 1; st.NextPos = 0; st.side = 0; st.notext = 0;
                        if (sp.force_left) {                                                   // Backtracking.h: right to left
                            st.qposL = (sp.partition[0] - 1) & 0xFFFF;
                            st.qposR = 0;
                        } else if (jv.bikmer_k && sp.u[s][0] == 0 && st.pev >= jv.bikmer_k && (jv.bikmer_base || jv.qflags[st.qidx] == 0)) {
                            // error-free first part: its first bikmer_k symbols (always searched to the right) in one lookup;
                            // the state is the one the error-free loop would have reached (SearchNg26.h:225-250)
                            uint32_t key = 0;
                            bool key_ok = true;
                            if (jv.bikmer_base) {
                                // generic layout: base-`bikmer_base` number of the symbols, first symbol = lowest digit
                                const uint8_t* qp = qsym + qoff[st.qidx] + st.qposR;
                                uint32_t mul = 1;
                                for (uint32_t p = 0; p < jv.bikmer_k; ++p) {
                                    const uint32_t c = __ldg(qp + p);
                                    if (c < first_symb || c >= ix.sigma) key_ok = false;
                                    key += (c - first_symb) * mul;
                                    mul *= jv.bikmer_base;
                                }
                            } else {
                                const uint64_t bit = 2 * (qoff[st.qidx] + st.qposR);
                                const uint32_t wi = (uint32_t)(bit >> 5);
                                key = __funnelshift_r(__ldg(jv.qpk + wi), __ldg(jv.qpk + wi + 1), (uint32_t)bit & 31u);
                                key &= (1u << (2 * jv.bikmer_k)) - 1u;
                            }
                            if (key_ok) {
                            const uint4 e = __ldg(jv.bikmer + key);
                            n_phys += 1;
                            n_ext += e.w >> 16;
                            n_look += e.w & 0xFFFFu;
                            st.lb = e.x; st.lb_rev = e.y; st.len = e.z;
                            st.steps = jv.bikmer_k;
                            st.qposR = (st.qposR + jv.bikmer_k) & 0xFFFF;
                            st.pev -= jv.bikmer_k;
                            st.mode = MODE_NOERR;
                            if (st.pev == 0) {                                                 // :241-249
                                st.part = 1;
                                st.pev = (np != 1) ? sp.partition[sp.pi[s][1]] : 0;
                                st.mode = MODE_NEXT;
                            }
                            const uint32_t lastq = __ldg(qsym + qoff[st.qidx] + ((st.qposR - 1) & 0xFFFF));
                            if (st.mode == MODE_NEXT) st.side = side_set(side_set(st.side, 1, 0, lastq), 1, 1, lastq);
                            }
                        }
                        if constexpr (ORDERED) {
                            rkey = order_key_root(sp, s);
                            // n rows of earlier searches of this query exist: this search cannot hold one of the first n
                            if (out.best_keys != nullptr && (rkey & (0xFFull << 56)) > prune_bound(out, st.qidx)) st.len = 0;
                        }
                        it = pack_item(st);
                    }
                }
                {
                    const uint32_t below = (1u << lane) - 1u;
                    const uint32_t bt = __ballot_sync(0xFFFFFFFFu, lane < got && to_text);
                    const uint32_t bc = __ballot_sync(0xFFFFFFFFu, lane < got && !to_text);
                    if (lane < got) {
                        if (to_text) {
                            stack[cap - 1 - (ttop + __popc(bt & below))] = it;
                        } else {
                            const uint32_t idx = top + __popc(bc & below);
                            stack[idx] = it;
                            if constexpr (ORDERED) kstack[idx] = rkey;
                        }
                    }
                    top += __popc(bc);
                    ttop += __popc(bt);
                    __syncwarp();
                    if (ttop >= 32) flush_text(32);
                }
            }
        }
        if (top == 0) {
            if (!more_roots) break;
            // progress: staged text items (ttop <= 31) leave only in groups of 32, so with nothing pending they alone can keep the
            // refill from having room for a round of roots.  Flushed, they leave top + ttop = 0, which every cap >= 32 (checked on
            // the host) admits: each iteration pops, pulls roots or ends.
            if (ttop + 32 > cap) flush_text(ttop);
            continue;
        }
        peak = top > peak ? top : peak;
        // ---- pop ---------------------------------------------------------------------------------------------
        const uint32_t nact = top < 32 ? top : 32;
        const bool active = lane < nact;
        State st;
        if (active) {
            st = unpack_item(stack[top - 1 - lane]);
            if constexpr (ORDERED) {
                st.key = kstack[top - 1 - lane];
                if (out.best_keys != nullptr && order_key_lower_bound<EDIT>(sp, st.key, st.steps, st.e) > prune_bound(out, st.qidx))
                    st.len = 0;                                  // every hit below this node comes after one already found: drop the subtree
            }
        }
        top -= nact;
        __syncwarp();

        // ---- expand: one node per lane and iteration; a lane whose node has exactly one child keeps going in
        //      registers (fast forward) instead of a round trip through the shared-memory stack ----------------
        unsigned long long cmask = 0;
        bool report = false;
        uint32_t q = 0, b0 = 0, b1 = 0, lo = 0, hi = 0, jrow = 0, jadd = 0, jlast = 0, jnoerr = 0, jlen = 16;
        typename OCC::Block blk0, blk1;
        bool is_single = false, noerr_cont = false;
        uint64_t qbase = 0;
        bool live = active;

        // one child of the expanded node (bit `bit` of cmask)
        auto make_child = [&](uint32_t bit) -> State {
            const uint32_t R = st.Right;
            const OCC& occ = ix.occ[R];
            State ch = st;
            ch.notext = 0;
            if (bit == 3) return ch;
            auto stepped = [&](uint32_t c) {
                uint32_t same, dother, clen;
                child_cursor(ix, occ, b0, b1, blk0, blk1, lo, hi, c, is_single, same, dother, clen);
                ch.len = clen;
                if (R) { ch.lb_rev = same; ch.lb = st.lb + dother; } else { ch.lb = same; ch.lb_rev = st.lb_rev + dother; }
                ch.steps = st.steps + 1;
            };
            if (bit == 0) {
                stepped(q);
                if (noerr_cont) {
                    if (R) ch.qposR = (st.qposR + 1) & 0xFFFF; else ch.qposL = (st.qposL - 1) & 0xFFFF;
                    ch.pev = st.pev - 1;
                    ch.NextPos = 0;
                    if (ch.pev > 0) {
                        ch.mode = MODE_NOERR;
                    } else {                                                                    // :241-249
                        ch.side = side_set(side_set(st.side, R, 0, q), R, 1, q);
                        ch.part = st.part + 1;
                        ch.pev = (ch.part != np) ? sp.partition[sp.pi[st.search][ch.part]] : 0;
                        if (R) ch.RInfo = INFO_M; else ch.LInfo = INFO_M;
                        ch.mode = MODE_NEXT;
                    }
                } else {                                                                        // match child
                    ch.side = side_set(side_set(st.side, R, 0, q), R, 1, q);
                    if (R) ch.RInfo = INFO_M; else ch.LInfo = INFO_M;
                    ch.NextPos = 1;
                    ch.mode = MODE_POS;
                }
            } else if (bit == 1) {                                                              // insertion: no index step
                if constexpr (ORDERED) ch.key = order_key_edge(sp, st.key, st.steps, st.e, is_single, 2 * ix.sigma + 1);
                ch.e = st.e + 1;
                ch.side = side_set(st.side, R, 1, q);
                if (R) ch.RInfo = INFO_I; else ch.LInfo = INFO_I;
                ch.NextPos = 1;
                ch.mode = MODE_POS;
            } else if (bit == 2) {                                                              // jlen symbols at once (len == 1)
                if (R) ch.lb_rev = jrow; else ch.lb = jrow;
                ch.steps = st.steps + jlen;
                ch.e = st.e + jadd;
                ch.side = side_set(side_set(st.side, R, 0, jlast), R, 1, jlast);
                if (st.mode == MODE_NOERR || jnoerr) {
                    // (jnoerr: a Hamming stretch that used up its error budget inside the window is in the error-free loop now)
                    if (R) ch.qposR = (st.qposR + jlen) & 0xFFFF; else ch.qposL = (st.qposL - jlen) & 0xFFFF;
                    ch.pev = st.pev - jlen;
                    ch.NextPos = 0;
                    ch.mode = MODE_NOERR;
                    if (ch.pev == 0) {
                        ch.part = st.part + 1;
                        ch.pev = (ch.part != np) ? sp.partition[sp.pi[st.search][ch.part]] : 0;
                        if (R) ch.RInfo = INFO_M; else ch.LInfo = INFO_M;
                        ch.mode = MODE_NEXT;
                    }
                } else {
                    // Hamming, errors allowed: jlen - 1 advances now, the last one is pending like after any match
                    if (R) ch.qposR = (st.qposR + jlen - 1) & 0xFFFF; else ch.qposL = (st.qposL - (jlen - 1)) & 0xFFFF;
                    ch.pev = st.pev - (jlen - 1);
                    if (R) ch.RInfo = INFO_M; else ch.LInfo = INFO_M;
                    ch.NextPos = 1;
                    ch.mode = MODE_POS;
                }
            } else {
                const bool is_sub = bit >= kSubBit;
                const uint32_t c = is_sub ? bit - kSubBit : bit - kDelBit;
                if constexpr (ORDERED)
                    ch.key = order_key_edge(sp, st.key, st.steps, st.e, false, is_single ? (is_sub ? 0u : 1u) : 2 * c + (is_sub ? 1u : 0u));
                stepped(c);
                ch.e = st.e + 1;
                ch.side = side_set(st.side, R, 0, c);
                ch.mode = MODE_POS;
                if (is_sub) {
                    ch.side = side_set(ch.side, R, 1, q);
                    if (R) ch.RInfo = INFO_S; else ch.LInfo = INFO_S;
                    ch.NextPos = 1;
                } else {
                    if (R) ch.RInfo = INFO_D; else ch.LInfo = INFO_D;
                    ch.NextPos = 0;
                }
            }
            return ch;
        };

        for (int ff = 0;; ++ff) {
            if (live) {
                cmask = 0;
                report = false;
                is_single = false;
                noerr_cont = false;
                bool go_dir = true;
                if (kText && ff > 0 && text_on && text_class(st, np, text_qflags, !OCC::kSymbolLoad)) {
                    // the node this lane fast-forwarded into belongs to the text kernel: it goes back as it is
                    cmask = CH_SELF;
                    go_dir = false;
                } else
                if (st.len == 0) {
                    go_dir = false;                                                                 // a root whose k-mer does not occur
                } else if (st.mode == MODE_POS) {                                                   // search_next_pos :119-141
                    if (st.NextPos) {
                        if (st.Right) st.qposR = (st.qposR + 1) & 0xFFFF; else st.qposL = (st.qposL - 1) & 0xFFFF;
                        st.pev -= 1;
                        if (st.pev == 0) {
                            st.part += 1;
                            if (st.part != np) st.pev = sp.partition[sp.pi[st.search][st.part]];
                            st.mode = MODE_NEXT;
                        }
                    }
                }
                if (cmask == 0 && st.len != 0 && st.mode == MODE_NEXT) {                            // search_next :98-117
                    if (st.part == np) {
                        bool ok = !EDIT || PSEUDO || ((st.LInfo == INFO_M || st.LInfo == INFO_I) && (st.RInfo == INFO_M || st.RInfo == INFO_I));
                        report = ok && sp.l[st.search][np - 1] <= st.e && st.e <= sp.u[st.search][np - 1];
                        go_dir = false;
                    } else {
                        st.Right = (st.part == 0) || (sp.pi[st.search][st.part - 1] < sp.pi[st.search][st.part]);
                        if (sp.force_left) st.Right = 0;
                    }
                }
                if (go_dir) {
                    const uint32_t R = st.Right;
                    const OCC& occ = ix.occ[R];
                    qbase = qoff[st.qidx];
                    lo = R ? st.lb_rev : st.lb;
                    hi = lo + st.len;
                    b0 = lo >> 6;
                    b1 = hi >> 6;
                    const uint32_t lp = sp.l[st.search][st.part], up = sp.u[st.search][st.part];
                    // ---- multi-symbol jump on a single-row interval.  DNA layout: LF^16 table, LF^4 for short stretches, 2-bit symbols
                    //      compared with the packed query; generic layout: LF^4 table with byte symbols compared with the raw query bytes ----
                    bool jumped = false;
                    uint32_t J = 0;                                   // symbols per jump
                    constexpr bool kBytes = OCC::kSymbolLoad;
                    constexpr uint32_t B = kBytes ? 8u : 2u;          // bits per symbol in a table entry
                    if (st.len == 1 && (kBytes ? jv.jump4[R] != nullptr : (jv.jump[R] != nullptr && jv.qflags[st.qidx] == 0))) {
                        const bool noerr = st.mode == MODE_NOERR;
                        const bool ham = !EDIT && !noerr && st.e < up;       // Hamming with errors left: the stretch must end inside the part
                        if (!kBytes && (noerr ? st.pev >= 16 : (ham && st.pev > 16))) J = 16;
                        else if (jv.jump4[R] != nullptr && (noerr ? st.pev >= 4 : (ham && st.pev > 4))) J = 4;
                    }
                    if (J) {
                        const uint2 e = __ldg(J == 16 ? jv.jump[R] + ((size_t)lo << jv.jshift[R]) : jv.jump4[R] + lo);
                        n_phys += 1;
                        if (e.x != kJumpInvalid) {
                            jumped = true;
                            const uint32_t W = B * J;                 // bits of the symbol word
                            // query symbols of the next J positions in walking direction, laid out like the table entry
                            uint32_t key;
                            if (kBytes) {
                                const uint8_t* qp = qsym + qbase + (R ? st.qposR : st.qposL - 3);
                                key = (uint32_t)__ldg(qp) | ((uint32_t)__ldg(qp + 1) << 8) | ((uint32_t)__ldg(qp + 2) << 16) | ((uint32_t)__ldg(qp + 3) << 24);
                            } else {
                                const uint64_t bit = 2 * (qbase + (R ? st.qposR : st.qposL - (J - 1)));
                                const uint32_t wi = (uint32_t)(bit >> 5);
                                key = __funnelshift_r(__ldg(jv.qpk + wi), __ldg(jv.qpk + wi + 1), (uint32_t)bit & 31u);
                                if (J != 16) key &= (1u << W) - 1u;
                            }
                            const uint32_t x = e.y ^ key;
                            uint32_t mm;                               // one bit per mismatching position, at the lowest bit of its field
                            if (kBytes) {
                                uint32_t y = x | (x >> 4);
                                y |= y >> 2;
                                y |= y >> 1;
                                mm = y & 0x01010101u;
                            } else {
                                mm = (x | (x >> 1)) & 0x55555555u;
                            }
                            const uint32_t budget = (st.mode == MODE_NOERR) ? 0u : up - st.e;   // mismatches this stretch may absorb (>= 1 when errors are left)
                            const uint32_t nm = __popc(mm);
                            // index (0..J-1, walking order: R from the low fields up, L from the high fields down) of the j-th mismatch, j = 1..
                            auto nth = [&](uint32_t j) -> int {
                                uint32_t m = mm;
                                int idx = -1;
                                for (uint32_t k = 0; k < j; ++k) {
                                    uint32_t pos = R ? (uint32_t)(__ffs(m) - 1) : 31u - (uint32_t)__clz(m);
                                    idx = R ? (int)(pos / B) : (int)(J - 1u - pos / B);
                                    m &= ~(1u << pos);
                                }
                                return idx;
                            };
                            // The counters follow the reference's walk over the same J positions: one extension per position; once
                            // the error budget of a Hamming stretch is used up it switches to its error-free loop at the next
                            // matching position, which repeats that extension (SearchNg26.h:311-315).
                            if (nm <= budget) {
                                cmask = CH_JUMP;
                                jrow = e.x;
                                jadd = nm;
                                jlen = J;
                                jlast = ((R ? key >> (W - B) : key) & ((1u << B) - 1u)) + (kBytes ? 0u : 1u);   // last query symbol consumed
                                jnoerr = 0;
                                uint32_t cnt = J;
                                if (st.mode != MODE_NOERR && nm == budget && nth(budget) < (int)J - 1) { jnoerr = 1; cnt += 1; }
                                n_ext += cnt; n_look += cnt;
                            } else {
                                const int d = nth(budget + 1);                               // the mismatch that ends the path
                                uint32_t cnt = (uint32_t)d + 1;
                                if (st.mode != MODE_NOERR && d - nth(budget) > 1) cnt += 1;
                                n_ext += cnt; n_look += cnt;
                            }
                        }
                    }
                    if (!jumped) {
                        q = __ldg(qsym + qbase + (R ? st.qposR : st.qposL));
                        if (st.mode == MODE_NOERR) {
                            noerr_cont = true;                                                          // search_next_dir_no_errors :225-250
                            if (q < ix.sigma) {
                                n_ext += 1; n_look += (b1 == b0) ? 1 : 2;      // algorithmic: two ranks, one or two blocks
                                if (st.len == 1) {
                                    // single row: it continues iff its own BWT symbol is q; one block serves symbol and rank
                                    is_single = true;
                                    blk0 = occ.load(b0, 0);
                                    blk1 = blk0;
                                    n_phys += 1;
                                    if (occ.symbol(blk0, lo) == q) cmask |= CH_MATCH;
                                } else {
                                    blk0 = occ.load(b0, q);
                                    blk1 = (b1 == b0) ? blk0 : occ.load(b1, q);
                                    n_phys += (b1 == b0) ? 1 : 2;
                                    uint32_t same, dother, clen;
                                    child_cursor(ix, occ, b0, b1, blk0, blk1, lo, hi, q, false, same, dother, clen);
                                    if (clen) cmask |= CH_MATCH;
                                }
                            }
                        } else {
                            const uint32_t TInfo = R ? st.RInfo : st.LInfo;
                            const uint32_t lastRank = side_get(st.side, R, 0), lastQRank = side_get(st.side, R, 1);
                            const bool Deletion = EDIT && (PSEUDO || (TInfo != INFO_S && TInfo != INFO_I));
                            const bool Insertion = EDIT && (PSEUDO || (TInfo != INFO_S && TInfo != INFO_D));
                            const bool matchAllowed = (st.pev > 1 || lp <= st.e) && st.e <= up && (PSEUDO || ((TInfo != INFO_I || q != lastQRank) && (TInfo != INFO_D || q != lastRank)));
                            const bool insAllowed = (st.pev > 1 || lp <= st.e + 1) && st.e + 1 <= up;
                            const bool mismatchAllowed = st.e + 1 <= up;
                            if (st.len > 1) {                                                           // search_next_dir :143-224
                                if (mismatchAllowed) {
                                    blk0 = occ.load(b0, 0);
                                    blk1 = (b1 == b0) ? blk0 : occ.load(b1, 0);
                                    n_ext += 1; n_look += (b1 == b0) ? 1 : 2; n_phys += (b1 == b0) ? 1 : 2;
                                    uint32_t same, dother, clen;
                                    if (matchAllowed && q < ix.sigma) {
                                        child_cursor(ix, occ, b0, b1, blk0, blk1, lo, hi, q, false, same, dother, clen);
                                        if (clen) cmask |= CH_MATCH;
                                    }
                                    for (uint32_t c = first_symb; c < ix.sigma; ++c) {
                                        child_cursor(ix, occ, b0, b1, blk0, blk1, lo, hi, c, false, same, dother, clen);
                                        if (!clen) continue;
                                        if (Deletion) cmask |= 1ull << (kDelBit + c);
                                        if (insAllowed && c != q) cmask |= 1ull << (kSubBit + c);
                                    }
                                    if (Insertion && insAllowed) cmask |= CH_INS;
                                } else if (matchAllowed) {
                                    noerr_cont = true;
                                    if (q < ix.sigma) {
                                        blk0 = occ.load(b0, q);
                                        blk1 = (b1 == b0) ? blk0 : occ.load(b1, q);
                                        n_ext += 1; n_look += (b1 == b0) ? 1 : 2; n_phys += (b1 == b0) ? 1 : 2;
                                        uint32_t same, dother, clen;
                                        child_cursor(ix, occ, b0, b1, blk0, blk1, lo, hi, q, false, same, dother, clen);
                                        if (clen) cmask |= CH_MATCH;
                                    }
                                }
                            } else {                                                                    // search_next_dir_single :251-365
                                is_single = true;
                                blk0 = occ.load(b0, 0);
                                blk1 = blk0;
                                n_ext += 1; n_look += 1; n_phys += 1;
                                const uint32_t single_sym = occ.symbol(blk0, lo);                       // symbolLeft/Right, BiFMIndexCursor.h:180-190
                                if (Insertion && insAllowed) cmask |= CH_INS;
                                if (single_sym >= first_symb) {
                                    if (single_sym == q) {
                                        if (matchAllowed) {
                                            if (!mismatchAllowed) {
                                                noerr_cont = true;
                                                n_ext += 1; n_look += 1;        // the reference's error-free loop repeats this extension (:311-315)
                                            }
                                            cmask |= CH_MATCH;
                                        }
                                        if (Deletion && mismatchAllowed) cmask |= 1ull << (kDelBit + single_sym);
                                    } else if (mismatchAllowed) {
                                        if (insAllowed) cmask |= 1ull << (kSubBit + single_sym);
                                        if (Deletion) cmask |= 1ull << (kDelBit + single_sym);
                                    }
                                }
                                // ---- window simulation of the error children -------------------------------------------------
                                // (sim_subtree_dies above): children whose whole subtree dies within the next 16 text symbols are
                                // accounted for -- their extensions are counted -- but never created.
                                const unsigned long long err_children = cmask & ~(CH_MATCH | CH_JUMP);
                                const uint2* sim_table = OCC::kSymbolLoad ? jv.jump4[R] : jv.jump[R];
                                if (EDIT && err_children && sim_table != nullptr && single_sym >= first_symb) {
                                    const uint2 je = __ldg(sim_table + (OCC::kSymbolLoad ? (size_t)lo : ((size_t)lo << jv.jshift[R])));
                                    n_phys += 1;
                                    if (je.x != kJumpInvalid) {
                                        // window in walking order, w[0] (= this row's symbol) in the low bits
                                        uint32_t window = je.y;
                                        if (!R) {                                   // direction 0 stores the nearest symbol in the high bits
                                            if (OCC::kSymbolLoad) {
                                                window = __byte_perm(window, 0, 0x0123);
                                            } else {
                                                window = __brev(window);
                                                window = ((window & 0xAAAAAAAAu) >> 1) | ((window & 0x55555555u) << 1);
                                            }
                                        }
                                        const uint8_t* qptr = qsym + qbase + (R ? st.qposR : st.qposL);
                                        unsigned long long rest = err_children;
                                        while (rest) {
                                            const uint32_t bit = __ffsll((long long)rest) - 1;
                                            rest &= rest - 1;
                                            SimState cs;
                                            cs.m = 1; cs.c = 0; cs.part = st.part; cs.pev = st.pev; cs.e = st.e + 1; cs.noerr = 0;
                                            cs.lastRank = lastRank; cs.lastQRank = lastQRank;
                                            bool ok = true;                      // false: the child's advance already leaves the window's reach
                                            bool adv = false;
                                            if (bit == 1) {                      // insertion: stays on this row
                                                cs.m = 0; cs.lastQRank = q; cs.T = INFO_I; adv = true;
                                            } else if (bit >= kSubBit) {         // substitution
                                                cs.lastRank = single_sym; cs.lastQRank = q; cs.T = INFO_S; adv = true;
                                            } else {                             // deletion: the query symbol is not consumed
                                                cs.lastRank = single_sym; cs.T = INFO_D;
                                            }
                                            if (adv) {
                                                cs.c = 1;
                                                cs.pev -= 1;
                                                if (cs.pev == 0) {
                                                    cs.part += 1;
                                                    if (cs.part == np) ok = false;
                                                    else {
                                                        const uint32_t nr = (sp.pi[st.search][cs.part - 1] < sp.pi[st.search][cs.part]) ? 1u : 0u;
                                                        if (sp.force_left || nr != R) ok = false;
                                                        else cs.pev = sp.partition[sp.pi[st.search][cs.part]];
                                                    }
                                                }
                                            }
                                            uint32_t sim_ext = 0;
                                            if (ok && sim_subtree_dies<EDIT, OCC::kSymbolLoad, PSEUDO>(sp, st.search, R, window, qptr, cs, sim_ext)) {
                                                cmask &= ~(1ull << bit);
                                                n_ext += sim_ext; n_look += sim_ext;
                                            }
                                        }
                                    }
                                }
                            }
                        }
                    }
                }
            }
            // fast forward: lanes with exactly one child (and nothing to report) continue with it
            const bool chain = live && !report && cmask != 0 && cmask != CH_SELF && (cmask & (cmask - 1)) == 0 && ff + 1 < kFastForward;
            // ... as long as enough lanes of the warp do so (the others idle meanwhile)
            if ((uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, chain)) < ff_min) break;
            if (chain) st = make_child((uint32_t)(__ffsll((long long)cmask) - 1));
            else live = false;
        }

        // ---- report leaves (warp aggregated append) -----------------------------------------------------------
        {
            uint32_t rb = __ballot_sync(0xFFFFFFFFu, report);
            if (rb) {
                unsigned long long base = 0;
                unsigned long long rows = report ? (unsigned long long)st.len : 0ull;
                for (int o = 16; o > 0; o >>= 1) rows += __shfl_xor_sync(0xFFFFFFFFu, rows, o);
                if (lane == (uint32_t)(__ffs(rb) - 1)) {
                    base = atomicAdd(out.hit_count, (unsigned long long)__popc(rb));
                    atomicAdd(out.row_count, rows);
                }
                base = __shfl_sync(0xFFFFFFFFu, base, __ffs(rb) - 1);
                if (report) {
                    unsigned long long idx = base + __popc(rb & ((1u << lane) - 1));
                    if (idx < out.hit_capacity) {
                        HitRec h;
                        h.qidx = st.qidx + out.qidx_base; h.lb = st.lb; h.lb_rev = sp.zero_lb_rev ? 0 : st.lb_rev; h.len = st.len; h.steps = st.steps; h.e = st.e;
                        out.hits[idx] = h;
                        if constexpr (ORDERED) {
                            out.hit_keys[idx] = st.key;
                            if (out.best_keys != nullptr) prune_insert(out, st.qidx, st.key, st.len);
                        }
                    }
                }
            }
        }

        if constexpr (kText) {
            // ---- push children, one round per child rank: a round's children are compacted by class with two ballots --------
            unsigned long long rest = cmask;
            const uint32_t below = (1u << lane) - 1u;
            for (;;) {
                const bool has = rest != 0;
                if (!__any_sync(0xFFFFFFFFu, has)) break;
                Item pk;
                bool tx = false;
                if (has) {
                    const uint32_t bit = __ffsll((long long)rest) - 1;
                    rest &= rest - 1;
                    const State c = make_child(bit);
                    tx = text_on && text_class(c, np, text_qflags, !OCC::kSymbolLoad);
                    pk = pack_item(c);
                }
                const uint32_t bt = __ballot_sync(0xFFFFFFFFu, has && tx), bc = __ballot_sync(0xFFFFFFFFu, has && !tx);
                const uint32_t nt = __popc(bt), nc = __popc(bc);
                if (top + ttop + nt + nc <= cap) {
                    if (has) stack[tx ? cap - 1 - (ttop + __popc(bt & below)) : top + __popc(bc & below)] = pk;
                    top += nc;
                    ttop += nt;
                    __syncwarp();
                    if (ttop >= 32) flush_text(32);
                } else {
                    // no room: the round goes to the global overflow list, which the host feeds to the next launch
                    unsigned long long base = 0;
                    if (lane == 0) base = atomicAdd(out.overflow_count, (unsigned long long)(nt + nc));
                    base = __shfl_sync(0xFFFFFFFFu, base, 0);
                    const unsigned long long idx = base + __popc((bt | bc) & below);
                    if (has && idx < out.overflow_capacity) out.overflow[idx] = pk;          // host sees overflow_count > capacity and fails loudly
                }
            }
        } else {
            // ---- compact + push children ---------------------------------------------------------------------------
            uint32_t nchild = __popcll(cmask);
            uint32_t incl = nchild;
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= (uint32_t)o) incl += v;
            }
            const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
            if (total == 0) continue;
            uint32_t slot = incl - nchild;
            Item* dst;
            unsigned long long* kdst = nullptr;
            bool drop = false;
            if (top + total <= cap) {
                dst = stack + top;
                if constexpr (ORDERED) kdst = kstack + top;
                top += total;
            } else {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(out.overflow_count, (unsigned long long)total);
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                dst = out.overflow + base;
                if constexpr (ORDERED) kdst = out.overflow_keys + base;
                drop = base + total > out.overflow_capacity;      // host sees overflow_count > capacity and fails loudly
            }
            if (cmask && !drop) {
                unsigned long long rest = cmask;
                while (rest) {
                    uint32_t bit = __ffsll((long long)rest) - 1;
                    rest &= rest - 1;
                    const State c = make_child(bit);
                    if constexpr (ORDERED) kdst[slot] = c.key;
                    dst[slot++] = pack_item(c);
                }
            }
            __syncwarp();
        }
    }
    if (ttop) flush_text(ttop);

    // ---- statistics ------------------------------------------------------------------------------------------
    for (int o = 16; o > 0; o >>= 1) {
        n_ext += __shfl_xor_sync(0xFFFFFFFFu, n_ext, o);
        n_look += __shfl_xor_sync(0xFFFFFFFFu, n_look, o);
        n_phys += __shfl_xor_sync(0xFFFFFFFFu, n_phys, o);
    }
    if (lane == 0) {
        atomicAdd(out.counters + CTR_EXTENSIONS, (unsigned long long)n_ext);
        atomicAdd(out.counters + CTR_OCC_LOOKUPS, (unsigned long long)n_look);
        atomicAdd(out.counters + CTR_LINE_REQUESTS, (unsigned long long)n_phys);
        atomicMax(out.counters + CTR_PEAK, (unsigned long long)peak);
    }
}

}  // namespace fmb
