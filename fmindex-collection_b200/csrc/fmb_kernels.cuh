// fmb_kernels.cuh -- sm_100a kernels: occ-table packing (K1), String_c / cursor batch ops, exact backward
// search (K2), LF-walk locate (K4), result compaction (K5).
#pragma once
#include "fmb_device.cuh"
#include "fmb_host.hpp"

namespace fmb {

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    uint64_t z = x + 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

// T[i] = 1 + (splitmix64(seed + i) >> 32) % (sigma-1), T[n-1] = 0   (fmb200.h fmb_synth_text_device)
__global__ void synth_text_kernel(uint8_t* text, uint64_t n, uint32_t sigma, uint64_t seed) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    text[i] = (i == n - 1) ? 0 : (uint8_t)(1 + (splitmix64(seed + i) >> 32) % (sigma - 1));
}

// reads[q*L + j] = text[off(q) + j], off(q) = splitmix64(q * 0x632BE59BD9B4E019 + seed) % (n - L)
__global__ void synth_reads_kernel(const uint8_t* __restrict__ text, uint64_t n, uint64_t nq, uint32_t L, uint64_t seed, uint8_t* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= nq * L) return;
    uint64_t q = i / L, j = i % L;
    uint64_t off = splitmix64(q * 0x632BE59BD9B4E019ull + seed) % (n - L);
    out[i] = text[off + j];
}

// locate-heavy workload (SURVEY.md §8d config C4): random text with a repeat family -- `copies` copies of a unit of
// `unit_len` symbols, each copy with `sub_per_mille`/1000 substituted symbols, placed in disjoint slots of n / copies
// symbols; queries are windows of the (unsubstituted) unit.
__device__ __forceinline__ uint8_t unit_symbol(uint64_t seed, uint32_t p, uint32_t sigma) {
    return (uint8_t)(1 + (splitmix64(seed * 0x2545F4914F6CDD1Dull + 0x1234567 + p) >> 32) % (sigma - 1));
}
__global__ void splice_repeats_kernel(uint8_t* __restrict__ text, uint64_t n, uint32_t sigma, uint64_t seed, uint32_t unit_len,
                                      uint32_t copies, uint32_t sub_per_mille) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= (uint64_t)copies * unit_len) return;
    uint32_t j = (uint32_t)(i / unit_len), p = (uint32_t)(i % unit_len);
    uint64_t slot = (n - 1) / copies;
    uint64_t at = j * slot + splitmix64(seed + 77 * j + 5) % (slot - unit_len) + p;
    uint8_t c = unit_symbol(seed, p, sigma);
    uint64_t h = splitmix64(seed + i * 0x9E3779B97F4A7C15ull + 99);
    if (h % 1000 < sub_per_mille) c = (uint8_t)(1 + (c - 1 + 1 + (h >> 20) % (sigma - 2)) % (sigma - 1));
    text[at] = c;
}
__global__ void unit_reads_kernel(uint64_t nq, uint32_t L, uint64_t seed, uint32_t unit_len, uint32_t sigma, uint8_t* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= nq * L) return;
    uint64_t q = i / L;
    uint32_t j = (uint32_t)(i % L);
    uint32_t u = (uint32_t)(splitmix64(q * 0x632BE59BD9B4E019ull + seed + 3) % (unit_len - L));
    out[i] = unit_symbol(seed, u + j, sigma);
}

// reads with planted errors (SURVEY.md §8d config C3, in the spirit of search/benchmark_bifmindex_searches.cpp:38-82 of the
// reference's tests): read q is copied from the text like synth_reads_kernel, then e = hash % (max_err+1) edits are applied
// one after the other: substitution (always a different symbol), insertion (last symbol dropped) or deletion (a random
// symbol appended); Hamming runs (edit == 0) plant substitutions only.  Length stays L.
__global__ void synth_reads_err_kernel(const uint8_t* __restrict__ text, uint64_t n, uint64_t nq, uint32_t L, uint64_t seed,
                                       uint32_t max_err, uint32_t edit, uint32_t sigma, uint8_t* __restrict__ out) {
    uint64_t q = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (q >= nq) return;
    uint64_t off = splitmix64(q * 0x632BE59BD9B4E019ull + seed) % (n - L);
    uint8_t r[512];
    for (uint32_t j = 0; j < L; ++j) r[j] = text[off + j];
    uint64_t h = splitmix64(q * 0x9E3779B97F4A7C15ull + seed * 31 + 7);
    uint32_t ne = (uint32_t)(h % (max_err + 1));
    for (uint32_t i = 0; i < ne; ++i) {
        h = splitmix64(h + i + 1);
        uint32_t kind = edit ? (uint32_t)(h % 3) : 0;
        uint32_t p = 1 + (uint32_t)((h >> 8) % (L - 2));
        uint32_t rnd = (uint32_t)((h >> 40) % (sigma - 1));
        if (kind == 0) {
            r[p] = (uint8_t)(1 + (r[p] - 1 + 1 + rnd % (sigma - 2)) % (sigma - 1));
        } else if (kind == 1) {
            for (uint32_t j = L - 1; j > p; --j) r[j] = r[j - 1];
            r[p] = (uint8_t)(1 + rnd);
        } else {
            for (uint32_t j = p; j + 1 < L; ++j) r[j] = r[j + 1];
            r[L - 1] = (uint8_t)(1 + rnd);
        }
    }
    for (uint32_t j = 0; j < L; ++j) out[q * L + j] = r[j];
}

// ---------------------------------------------------------------------------------------------------------
// K1: pack 64 BWT bytes into one DnaBlock (local counts; absolute counts are added after a scan)
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_dna_kernel(const uint8_t* __restrict__ bwt, uint64_t n, uint32_t sigma,
                                                       DnaBlock* __restrict__ blocks, uint4* __restrict__ counts,
                                                       uint32_t* __restrict__ dcount, uint32_t* __restrict__ bad) {
    uint64_t blk = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    uint64_t nblocks = n / 64 + 1;
    if (blk > nblocks) return;
    if (blk == nblocks) { dcount[blk] = 0; return; }
    uint64_t base = blk * 64;
    uint64_t p0 = 0, p1 = 0;
    uint32_t c[4] = {0, 0, 0, 0};
    uint32_t nd = 0, isbad = 0;
    if (base + 64 <= n && (reinterpret_cast<uintptr_t>(bwt) & 15) == 0) {
        const uint4* src = reinterpret_cast<const uint4*>(bwt + base);
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            uint4 v = __ldg(src + w);
            uint32_t words[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    uint32_t s = (words[j] >> (8 * b)) & 0xFF;
                    uint32_t r = w * 16 + j * 4 + b;
                    isbad |= (s >= sigma);
                    uint32_t k = s ? s - 1 : 0;
                    nd += (s == 0);
                    p0 |= (uint64_t)(k & 1) << r;
                    p1 |= (uint64_t)((k >> 1) & 1) << r;
                    c[0] += (s == 1); c[1] += (s == 2); c[2] += (s == 3); c[3] += (s == 4);
                }
            }
        }
    } else {
        for (uint32_t r = 0; r < 64 && base + r < n; ++r) {
            uint32_t s = bwt[base + r];
            isbad |= (s >= sigma);
            uint32_t k = s ? s - 1 : 0;
            nd += (s == 0);
            p0 |= (uint64_t)(k & 1) << r;
            p1 |= (uint64_t)((k >> 1) & 1) << r;
            c[0] += (s == 1); c[1] += (s == 2); c[2] += (s == 3); c[3] += (s == 4);
        }
    }
    DnaBlock out;
    out.cnt[0] = out.cnt[1] = out.cnt[2] = out.cnt[3] = 0;
    out.p0 = p0;
    out.p1 = p1;
    blocks[blk] = out;
    counts[blk] = make_uint4(c[0], c[1], c[2], c[3]);
    dcount[blk] = nd;
    if (isbad) atomicOr(bad, 1u);
}

__global__ void store_counts_kernel(DnaBlock* __restrict__ blocks, const uint4* __restrict__ counts, uint64_t nblocks) {
    uint64_t blk = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (blk >= nblocks) return;
    uint4 c = counts[blk];
    *reinterpret_cast<uint4*>(blocks + blk) = c;
}

__global__ void scatter_delims_kernel(const uint8_t* __restrict__ bwt, uint64_t n, const uint32_t* __restrict__ dstart,
                                      uint32_t* __restrict__ delim_rows) {
    uint64_t blk = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    uint64_t nblocks = n / 64 + 1;
    if (blk >= nblocks) return;
    uint32_t a = dstart[blk], b = dstart[blk + 1];
    if (a == b) return;
    uint64_t base = blk * 64;
    for (uint32_t r = 0; r < 64 && base + r < n; ++r)
        if (bwt[base + r] == 0) delim_rows[a++] = (uint32_t)(base + r);
}

// ---------------------------------------------------------------------------------------------------------
// K1 (generic layout, 5 < sigma <= 32): per 64 rows the bit planes + local symbol counts; after an exclusive scan of the
// counts the block receives its sigma-1 exclusive prefix counts pc[c-1] = # symbols < c before the block.
// ---------------------------------------------------------------------------------------------------------
struct Cnt32 {
    uint32_t c[32];
};
struct Cnt32Add {
    __host__ __device__ Cnt32 operator()(const Cnt32& a, const Cnt32& b) const {
        Cnt32 r;
#pragma unroll
        for (int i = 0; i < 32; ++i) r.c[i] = a.c[i] + b.c[i];
        return r;
    }
};
__global__ void __launch_bounds__(128) pack_gen_kernel(const uint8_t* __restrict__ bwt, uint64_t n, uint32_t sigma, uint32_t planes, uint32_t stride,
                                                       uint8_t* __restrict__ blocks, Cnt32* __restrict__ counts, uint32_t* __restrict__ bad) {
    uint64_t blk = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    uint64_t nblocks = n / 64 + 1;
    if (blk >= nblocks) return;
    uint64_t base = blk * 64;
    uint64_t pl[5] = {0, 0, 0, 0, 0};
    Cnt32 c;
#pragma unroll
    for (int i = 0; i < 32; ++i) c.c[i] = 0;
    uint32_t isbad = 0;
    for (uint32_t r = 0; r < 64 && base + r < n; ++r) {
        uint32_t s = bwt[base + r];
        if (s >= sigma) { isbad = 1; s = 0; }
#pragma unroll
        for (int i = 0; i < 32; ++i) c.c[i] += (s == (uint32_t)i);
#pragma unroll
        for (int j = 0; j < 5; ++j) pl[j] |= (uint64_t)((s >> j) & 1) << r;
    }
    uint64_t* out = reinterpret_cast<uint64_t*>(blocks + blk * stride);
    for (uint32_t j = 0; j < planes; ++j) out[j] = pl[j];
    counts[blk] = c;
    if (isbad) atomicOr(bad, 1u);
}
__global__ void store_gen_counts_kernel(uint8_t* __restrict__ blocks, uint32_t stride, uint32_t planes, uint32_t sigma, const Cnt32* __restrict__ counts,
                                        uint64_t nblocks) {
    uint64_t blk = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (blk >= nblocks) return;
    uint32_t* pc = reinterpret_cast<uint32_t*>(blocks + blk * stride + 8 * planes);
    const Cnt32& c = counts[blk];
    uint32_t acc = 0;
    for (uint32_t s = 0; s + 1 < sigma; ++s) {
        acc += c.c[s];
        pc[s] = acc;                       // # symbols <= s = # symbols < s+1 before the block
    }
}

template <class OCC>
__global__ void compute_C_kernel(IndexView<OCC> ix, uint64_t* out) {
    uint32_t s = threadIdx.x;
    if (s > ix.sigma) return;
    const OCC& occ = ix.occ[0];
    typename OCC::Block b = occ.load(ix.n >> 6, s < ix.sigma ? s : ix.sigma - 1);
    // prefix_rank(n, s); for s == sigma everything is smaller
    out[s] = (s == ix.sigma) ? ix.n : occ.prefix_rank(b, ix.n, s);
}

__global__ void popcount_words_kernel(const uint64_t* __restrict__ bitmap, uint64_t have, uint64_t count, uint32_t* __restrict__ out) {
    uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (w >= count) return;
    out[w] = w < have ? __popcll(bitmap[w]) : 0;
}
__global__ void build_marks_kernel(const uint64_t* __restrict__ bitmap, uint64_t have, uint64_t words,
                                   const uint32_t* __restrict__ before, uint4* __restrict__ marks) {
    uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (w >= words) return;
    uint64_t bits = w < have ? bitmap[w] : 0;
    marks[w] = make_uint4((uint32_t)bits, (uint32_t)(bits >> 32), before[w], 0);
}
__global__ void export_marks_kernel(const uint4* __restrict__ marks, uint64_t have, uint64_t* __restrict__ out) {
    uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (w >= have) return;
    uint4 m = marks[w];
    out[w] = (uint64_t)m.x | ((uint64_t)m.y << 32);
}
__global__ void zip_samples_kernel(const uint32_t* __restrict__ seq, const uint32_t* __restrict__ pos, uint64_t count, uint2* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    out[i] = make_uint2(seq[i], pos[i]);
}

template <class OCC>
__global__ void unpack_bwt_kernel(IndexView<OCC> ix, int dir, uint8_t* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= ix.n) return;
    const OCC& occ = ix.occ[dir];
    typename OCC::Block b = occ.load((uint32_t)(i >> 6), 0);
    out[i] = (uint8_t)occ.symbol(b, (row_t)i);
}

// ---------------------------------------------------------------------------------------------------------
// String_c batch ops: op 0 symbol, 1 rank, 2 prefix_rank, 3 all_ranks_and_prefix_ranks
// (string/concepts.h:48-87; all_ranks_and_prefix_ranks: prs[0] = 0, prs[c] = prs[c-1] + rs[c-1],
//  string/InterleavedBitvector.h:141-160)
// ---------------------------------------------------------------------------------------------------------
template <class OCC>
__global__ void string_op_kernel(IndexView<OCC> ix, int dir, int op, const uint64_t* __restrict__ idx,
                                 const uint8_t* __restrict__ symb, uint64_t count, uint64_t* __restrict__ out,
                                 uint64_t* __restrict__ out2) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    const OCC& occ = ix.occ[dir];
    row_t row = (row_t)idx[i];
    if (op == 0) {
        typename OCC::Block b = occ.load(row >> 6, 0);
        out[i] = occ.symbol(b, row);
    } else if (op == 1) {
        typename OCC::Block b = occ.load(row >> 6, symb[i]);
        out[i] = occ.rank(b, row, symb[i]);
    } else if (op == 2) {
        uint32_t s = symb[i];
        if (s >= ix.sigma) { out[i] = row; return; }
        typename OCC::Block b = occ.load(row >> 6, s);
        out[i] = occ.prefix_rank(b, row, s);
    } else {
        uint64_t acc = 0;
        for (uint32_t s = 0; s < ix.sigma; ++s) {
            typename OCC::Block b = occ.load(row >> 6, s);
            uint64_t r = occ.rank(b, row, s);
            out[i * ix.sigma + s] = r;
            out2[i * ix.sigma + s] = acc;
            acc += r;
        }
    }
}

// cursor batch ops (fmindex/BiFMIndexCursor.h:113-128; :58-82 for all symbols)
template <class OCC>
__global__ void cursor_op_kernel(IndexView<OCC> ix, int right, int all, const uint64_t* __restrict__ cur,
                                 const uint8_t* __restrict__ symb, uint64_t count, uint64_t* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    Cursor c{(row_t)cur[4 * i], (row_t)cur[4 * i + 1], (row_t)cur[4 * i + 2], (uint32_t)cur[4 * i + 3]};
    uint32_t lookups = 0;
    if (!all) {
        Cursor o = extend_bi(ix, c, symb[i], right, lookups);
        out[4 * i] = o.lb; out[4 * i + 1] = o.lb_rev; out[4 * i + 2] = o.len; out[4 * i + 3] = o.steps;
    } else {
        for (uint32_t s = 0; s < ix.sigma; ++s) {
            Cursor o = extend_bi(ix, c, s, right, lookups);
            uint64_t* p = out + (i * ix.sigma + s) * 4;
            p[0] = o.lb; p[1] = o.lb_rev; p[2] = o.len; p[3] = o.steps;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// K2: exact backward search, one query per thread, full occupancy (search/SearchNoErrors.h:13-26 per query).
// The reference keeps 32 queries in flight per core in software (:29-85); here every resident thread is one
// in-flight query: 2048 per SM, ~300 k per GPU, which is what hides the ~1 us random-sector latency.
// Query symbols are read as aligned 16-byte chunks (register buffered, one load per 16 steps).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t chunk_byte(const uint4& v, uint32_t i) {
    uint32_t w = (i & 8) ? ((i & 4) ? v.w : v.z) : ((i & 4) ? v.y : v.x);
    return (w >> (8 * (i & 3))) & 0xFF;
}

template <class OCC>
__global__ void __launch_bounds__(256) exact_search_kernel(const __grid_constant__ IndexView<OCC> ix, const uint8_t* __restrict__ qsym,
                                                           const uint64_t* __restrict__ qoff, uint32_t nq, uint32_t qidx_base,
                                                           HitRec* __restrict__ out_hits, uint32_t* __restrict__ out_len,
                                                           unsigned long long* __restrict__ counters, const uint2* __restrict__ jump4) {
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t ext = 0, lookups = 0, found = 0;
    unsigned long long rows = 0;
    if (q < nq) {
        uint64_t off = qoff[q];
        uint32_t L = (uint32_t)(qoff[q + 1] - off);
        row_t lb = 0, len = ix.n;
        uint64_t cur_chunk = ~uint64_t(0);
        uint4 chunk = make_uint4(0, 0, 0, 0);
        auto byte_at = [&](uint32_t pos) -> uint32_t {
            uint64_t a = off + pos;
            if ((a >> 4) != cur_chunk) {
                cur_chunk = a >> 4;
                chunk = __ldg(reinterpret_cast<const uint4*>(qsym) + cur_chunk);
            }
            return chunk_byte(chunk, (uint32_t)(a & 15));
        };
        for (uint32_t pos = L; pos > 0;) {
            if (OCC::kSymbolLoad && len == 1 && pos >= 4 && jump4 != nullptr) {
                // generic layout: four symbols per lookup on a single-row interval (LF^4 table with byte symbols, farthest symbol
                // in the low byte = query order).  The DNA instantiation of this kernel is the exact-counting one and never jumps.
                const uint2 e = __ldg(jump4 + lb);
                if (e.x != kJumpInvalid) {
                    const uint32_t key = byte_at(pos - 4) | (byte_at(pos - 3) << 8) | (byte_at(pos - 2) << 16) | (byte_at(pos - 1) << 24);
                    ext += 4; lookups += 4;
                    if (e.y != key) { len = 0; break; }
                    lb = e.x;
                    pos -= 4;
                    continue;
                }
            }
            --pos;
            uint32_t c = byte_at(pos);
            if (c >= ix.sigma) { len = 0; break; }
            extend_left_uni(ix, lb, len, c, lookups);
            ++ext;
            if (len == 0) break;
        }
        HitRec h;
        h.qidx = q + qidx_base; h.lb = lb; h.lb_rev = 0; h.len = len; h.steps = L; h.e = 0;
        out_hits[q] = h;
        out_len[q] = len;
        found = len ? 1u : 0u;
        rows = len;
    }
    // [0] extensions, [1] occ lookups; [4] hits, [5] rows of all hits
    block_count2(counters, 0, ext, 1, lookups);
    block_count3(counters, 4, found, 4, 0, 5, rows);
}

// ---------------------------------------------------------------------------------------------------------
// K1b: two-symbol table (OccDna2, fmb_device.cuh).  Built from the one-symbol table itself:
//      y = BWT[i],  x = BWT[LF(i)]  with LF(i) = C[y] + rank(i, y);  code = (y-1)*4 + (x-1), 0xFF = special row.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pair_codes_kernel(const __grid_constant__ IndexView<OccDna> ix, int dir, uint8_t* __restrict__ codes) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= ix.n) return;
    const OccDna& occ = ix.occ[dir];
    DnaBlock b = occ.load((uint32_t)(i >> 6));
    uint32_t y = occ.symbol(b, (row_t)i);
    uint8_t code = 0xFF;
    if (y != 0) {
        row_t j = ix.C[y] + occ.rank(b, (row_t)i, y);
        DnaBlock b2 = occ.load(j >> 6);
        uint32_t x = occ.symbol(b2, j);
        if (x != 0) code = (uint8_t)((y - 1) * 4 + (x - 1));
    }
    codes[i] = code;
}

struct Cnt16 {
    uint32_t c[16];
};
struct Cnt16Add {
    __host__ __device__ Cnt16 operator()(const Cnt16& a, const Cnt16& b) const {
        Cnt16 r;
#pragma unroll
        for (int i = 0; i < 16; ++i) r.c[i] = a.c[i] + b.c[i];
        return r;
    }
};

// one thread per quarter (32 rows): planes + local counts of its rows
__global__ void __launch_bounds__(256) pack_pairs_kernel(const uint8_t* __restrict__ codes, uint64_t n, uint64_t nblocks,
                                                         uint4* __restrict__ lines, uint32_t* __restrict__ qcounts /*[nblocks*4][16]*/,
                                                         uint32_t* __restrict__ special_count /*[nblocks*4 + 1]*/) {
    uint64_t qd = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;      // quarter index
    if (qd > nblocks * 4) return;
    if (qd == nblocks * 4) { special_count[qd] = 0; return; }
    uint64_t base = qd * 32;
    uint32_t pl[4] = {0, 0, 0, 0};
    uint32_t cnt[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) cnt[i] = 0;
    uint32_t ns = 0;
    for (uint32_t r = 0; r < 32 && base + r < n; ++r) {
        uint32_t c = codes[base + r];
        if (c == 0xFF) { ++ns; c = 0; }
#pragma unroll
        for (int i = 0; i < 16; ++i) cnt[i] += (c == (uint32_t)i);
        pl[0] |= (c & 1) << r;
        pl[1] |= ((c >> 1) & 1) << r;
        pl[2] |= ((c >> 2) & 1) << r;
        pl[3] |= ((c >> 3) & 1) << r;
    }
    lines[qd * 2 + 1] = make_uint4(pl[0], pl[1], pl[2], pl[3]);
#pragma unroll
    for (int i = 0; i < 16; ++i) qcounts[qd * 16 + i] = cnt[i];
    special_count[qd] = ns;
}
// per block: sum of its four quarters
__global__ void block_counts_kernel(const uint32_t* __restrict__ qcounts, uint64_t nblocks, Cnt16* __restrict__ bcounts) {
    uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= nblocks * 16) return;
    uint64_t blk = t >> 4;
    uint32_t i = t & 15;
    const uint32_t* q = qcounts + blk * 64;
    bcounts[blk].c[i] = q[i] + q[16 + i] + q[32 + i] + q[48 + i];
}
// after the exclusive scan: quarter k of block b receives the absolute counters 4k .. 4k+3
__global__ void store_pair_counts_kernel(uint4* __restrict__ lines, const Cnt16* __restrict__ bcounts, uint64_t nblocks) {
    uint64_t qd = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (qd >= nblocks * 4) return;
    const Cnt16& c = bcounts[qd >> 2];
    uint32_t k = (qd & 3) * 4;
    lines[qd * 2] = make_uint4(c.c[k], c.c[k + 1], c.c[k + 2], c.c[k + 3]);
}
__global__ void scatter_specials_kernel(const uint8_t* __restrict__ codes, uint64_t n, uint64_t nquarters, const uint32_t* __restrict__ start,
                                        uint32_t* __restrict__ specials) {
    uint64_t qd = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (qd >= nquarters) return;
    uint32_t a = start[qd], b = start[qd + 1];
    if (a == b) return;
    uint64_t base = qd * 32;
    for (uint32_t r = 0; r < 32 && base + r < n; ++r)
        if (codes[base + r] == 0xFF) specials[a++] = (uint32_t)(base + r);
}

// (lb, len) of every k-mer: thread i searches the pattern whose symbol at position p (from the left) is ((i >> 2p) & 3) + 1,
// i.e. the index is the 2-bit packed pattern in the order the packed query stream stores it
__global__ void __launch_bounds__(256) kmer_table_kernel(const __grid_constant__ IndexView<OccDna> ix, uint32_t k, uint64_t count, uint2* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    row_t lb = 0, len = ix.n;
    uint32_t dummy = 0;
    for (uint32_t p = k; p-- > 0 && len;) extend_left_uni(ix, lb, len, (uint32_t)((i >> (2 * p)) & 3) + 1, dummy);
    out[i] = make_uint2(lb, len);
}

__global__ void iota_offsets_kernel(uint64_t* __restrict__ off, uint64_t count, uint32_t stride) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < count) off[i] = i * stride;
}
__global__ void rebase_offsets_kernel(uint64_t* __restrict__ off, uint64_t count, uint64_t base) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < count) off[i] -= base;
}

// Reverse-complement doubling of a query batch on the device (the example's loadQueries pushes every read followed by its reverse
// complement, example/utils.h:62-74): query i of the uploaded batch becomes query 2i (unchanged) and query 2i+1 (reversed, every
// symbol mapped through `comp`).  One warp per uploaded query; offsets are relative to the first symbol of the batch.
struct ComplementTable { uint8_t map[32]; };
__global__ void __launch_bounds__(256) revcomp_double_kernel(const uint8_t* __restrict__ fwd, const uint64_t* __restrict__ foff, uint64_t nq,
                                                             const __grid_constant__ ComplementTable comp, uint8_t* __restrict__ out,
                                                             uint64_t* __restrict__ ooff) {
    const uint64_t w = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (w >= nq) return;
    const uint64_t b = foff[w], e = foff[w + 1], L = e - b;
    if (lane == 0) {
        ooff[2 * w] = 2 * b;
        ooff[2 * w + 1] = 2 * b + L;
        if (w + 1 == nq) ooff[2 * nq] = 2 * e;
    }
    for (uint64_t j = lane; j < L; j += 32) {
        const uint8_t c = fwd[b + j];
        out[2 * b + j] = c;
        out[2 * b + L + (L - 1 - j)] = c < 32 ? comp.map[c] : c;
    }
}

// bidirectional k-mer table (fmb_scheme.cuh JumpView::bikmer): k extendRight steps per pattern, with the work the
// reference's error-free loop spends on them
__global__ void __launch_bounds__(256) bikmer_table_kernel(const __grid_constant__ IndexView<OccDna> ix, uint32_t k, uint64_t count, uint4* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    Cursor c{0, 0, ix.n, 0};
    uint32_t ext = 0, look = 0;
    for (uint32_t p = 0; p < k && c.len; ++p) {
        c = extend_bi(ix, c, (uint32_t)((i >> (2 * p)) & 3) + 1, 1, look);
        ++ext;
    }
    out[i] = make_uint4(c.lb, c.lb_rev, c.len, (ext << 16) | look);
}

// the same for the generic layout: pattern i has the symbols first_symb + digit_p(i) in base (sigma - first_symb), first symbol = lowest digit
template <class OCC>
__global__ void __launch_bounds__(256) bikmer_table_gen_kernel(const __grid_constant__ IndexView<OCC> ix, uint32_t k, uint32_t base, uint64_t count,
                                                               uint4* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    Cursor c{0, 0, ix.n, 0};
    uint32_t ext = 0, look = 0;
    uint64_t rest = i;
    for (uint32_t p = 0; p < k && c.len; ++p) {
        c = extend_bi(ix, c, ix.first_symb + (uint32_t)(rest % base), 1, look);
        rest /= base;
        ++ext;
    }
    out[i] = make_uint4(c.lb, c.lb_rev, c.len, (ext << 16) | look);
}

// 2-bit packing of the query symbols (symbol-1, 16 symbols per word, first symbol in the low bits).  Queries holding a
// symbol that has no 2-bit code (0 or >= sigma) are flagged and take the byte path of the search kernel.
__device__ __forceinline__ uint32_t pack4(uint32_t w, uint32_t sigma, bool& bad) {
    // code = (byte - 1) & 3 = (byte + 3) & 3, added per byte without carries into the neighbour (which may belong to
    // another query): bit 7 is masked off first, it does not reach the two low bits
    uint32_t v = ((w & 0x7F7F7F7Fu) + 0x03030303u) & 0x03030303u;
    const uint32_t lim = sigma - 1;                    // valid bytes: 1 .. sigma-1  <=>  (byte - 1) < sigma - 1 (unsigned)
    bad = bad || ((w & 0xFF) - 1u >= lim) || (((w >> 8) & 0xFF) - 1u >= lim) || (((w >> 16) & 0xFF) - 1u >= lim) || ((w >> 24) - 1u >= lim);
    return (v * 0x00041041u >> 18) & 0xFFu;            // gathers the four 2-bit fields (disjoint partial products)
}
__global__ void __launch_bounds__(256) pack_queries_kernel(const uint8_t* __restrict__ qsym, uint64_t total, const uint64_t* __restrict__ qoff,
                                                           uint64_t nq, uint32_t sigma, uint32_t* __restrict__ packed, uint64_t words,
                                                           uint8_t* __restrict__ qflags) {
    uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (w >= words) return;
    uint4 c = __ldg(reinterpret_cast<const uint4*>(qsym) + w);         // the symbol buffer is padded with 0xFF
    bool bad = false;
    uint32_t out = pack4(c.x, sigma, bad) | (pack4(c.y, sigma, bad) << 8) | (pack4(c.z, sigma, bad) << 16) | (pack4(c.w, sigma, bad) << 24);
    packed[w] = out;
    if (bad) {
        // rare: flag every query owning an uncodable symbol of this word
        uint32_t words4[4] = {c.x, c.y, c.z, c.w};
        for (uint32_t i = 0; i < 16; ++i) {
            uint64_t at = w * 16 + i;
            if (at >= total) break;
            uint32_t b = (words4[i >> 2] >> (8 * (i & 3))) & 0xFF;
            if (b >= 1 && b < sigma) continue;
            uint64_t lo = 0, hi = nq;                                   // last query with qoff[q] <= at
            while (hi - lo > 1) {
                uint64_t mid = (lo + hi) >> 1;
                if (qoff[mid] <= at) lo = mid; else hi = mid;
            }
            qflags[lo] = 1;
        }
    }
}

// 2-bit packed host queries -> byte symbols (fmb_queries_upload_packed): thread t writes the 16 symbols [16 t, 16 t + 16) of the slice;
// symbol i of the slice is the 2-bit field `shift + i` of the word stream (shift < 16: the slice may start inside a word)
__global__ void __launch_bounds__(256) unpack_queries_kernel(const uint32_t* __restrict__ words, uint64_t shift, uint64_t total, uint8_t* __restrict__ out) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t * 16 >= total) return;
    const uint64_t bit = 2 * (shift + t * 16);
    const uint64_t wi = bit >> 5;
    const uint32_t lo = words[wi], hi = (bit & 31u) ? words[wi + 1] : 0u;      // the second word exists whenever it is needed
    const uint32_t v = __funnelshift_r(lo, hi, (uint32_t)bit & 31u);
    for (uint32_t i = 0; i < 16 && t * 16 + i < total; ++i) out[t * 16 + i] = (uint8_t)(((v >> (2 * i)) & 3u) + 1u);
}
// symbols without 2-bit code (the delimiter, anything >= sigma): listed by position in the whole batch
__global__ void apply_exceptions_kernel(const uint64_t* __restrict__ pos, const uint8_t* __restrict__ sym, uint64_t count, uint64_t first, uint8_t* __restrict__ out) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < count) out[pos[i] - first] = sym[i];
}

// LF^16 jump table by pointer doubling: J1[row] = {LF(row), BWT[row]-1};  J2k[row] = {J_k[J_k[row].x].x, syms << 2k | syms'}
// (the farthest symbol ends up in the low bits: the order of the 2-bit packed query stream)
// DNA layout: 2-bit codes (symbol - 1); generic layout: the symbol itself in 8 bits (compared with the raw query bytes)
template <class OCC>
__global__ void __launch_bounds__(256) jump_init_kernel(const __grid_constant__ IndexView<OCC> ix, int dir, uint2* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= ix.n) return;
    const OCC& occ = ix.occ[dir];
    typename OCC::Block b = occ.load((uint32_t)(i >> 6), 0);
    uint32_t y = occ.symbol(b, (row_t)i);
    if (y < ix.first_symb) { out[i] = make_uint2(kJumpInvalid, 0); return; }      // a delimiter: nothing jumps across it
    if (OCC::kSymbolLoad) b = occ.load((uint32_t)(i >> 6), y);
    out[i] = make_uint2(ix.C[y] + occ.rank(b, (row_t)i, y), OCC::kSymbolLoad ? y : y - 1);
}
__global__ void __launch_bounds__(256) jump_double_kernel(const uint2* __restrict__ in, uint2* __restrict__ out, uint64_t n, uint32_t shift, int nearest_low) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint2 a = in[i];
    uint2 r = make_uint2(kJumpInvalid, 0);
    if (a.x != kJumpInvalid) {
        uint2 b = __ldg(in + a.x);
        // a = the nearer `shift/2` symbols, b = the farther ones
        if (b.x != kJumpInvalid) r = make_uint2(b.x, nearest_low ? (a.y | (b.y << shift)) : ((a.y << shift) | b.y));
    }
    out[i] = r;
}

// merged LF^16 / LF^32 table: out[row] = {J16[row], J16[J16[row].x]} (16 bytes per row)
__global__ void __launch_bounds__(256) jump_widen_kernel(const uint2* __restrict__ in, uint4* __restrict__ out, uint64_t n) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint2 a = in[i];
    uint2 b = make_uint2(kJumpInvalid, 0);
    if (a.x != kJumpInvalid) b = __ldg(in + a.x);
    out[i] = make_uint4(a.x, a.y, b.x, b.y);
}

// ---------------------------------------------------------------------------------------------------------
// K2b: exact backward search with two-symbol steps.  A group of 4 lanes owns one query: every lane fetches one
// 32-byte quarter of the 128-byte line (ONE request per line for the memory system), computes its share of the
// two ranks and the group adds them up with 2 SHFL.XOR each.  All 4 lanes keep the (identical) query state, so no
// broadcast is needed.  Pairs containing the delimiter symbol 0 and the odd leading symbol take one-symbol steps on
// the 32-byte table (all lanes of the group read the same sector = one request).
// Results are identical to exact_search_kernel: the final (lb, len) of a pattern does not depend on the step width.
// 8 blocks per SM: 32 registers, 2048 resident threads per SM.
// Text check (Occ2View::isa): a single-row interval with at least kTextCheckMin symbols left is decided on the text instead of the LF
// jumps; out_at (may be nullptr) receives the (seq, pos) of such hits for locate, kNoSeq for every other query.
// ---------------------------------------------------------------------------------------------------------
constexpr uint32_t kTextCheckMin = 16;
__global__ void __launch_bounds__(256, 8) exact_search2_kernel(const __grid_constant__ IndexView<OccDna> ix, const __grid_constant__ Occ2View o2,
                                                                  const uint8_t* __restrict__ qsym, const uint32_t* __restrict__ qpk,
                                                                  const uint8_t* __restrict__ qflags, const uint64_t* __restrict__ qoff, uint32_t nq,
                                                                  uint32_t qidx_base, HitRec* __restrict__ out_hits, uint32_t* __restrict__ out_len,
                                                                  uint2* __restrict__ out_at, unsigned long long* __restrict__ counters) {
    const uint32_t q = (uint32_t)((blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 2);      // 4 lanes per query: the thread index may exceed 32 bits
    const uint32_t sub = threadIdx.x & 3;
    const uint32_t gmask = 0xFu << (threadIdx.x & 28);
    uint32_t lines = 0, found = 0;
    unsigned long long rows = 0;
    bool checked = false;
    if (q < nq) {
        const uint64_t off = qoff[q];
        const uint32_t L = (uint32_t)(qoff[q + 1] - off);
        row_t lb = 0, len = ix.n;
        uint32_t dummy = 0;
        if (qflags[q]) {
            // byte path: the query holds a delimiter or an out-of-range symbol -> one-symbol steps, reference semantics
            for (uint32_t pos = L; pos-- > 0 && len;) {
                uint32_t c = __ldg(qsym + off + pos);
                if (c >= ix.sigma) { len = 0; break; }
                extend_left_uni(ix, lb, len, c, dummy);
                lines += 1;
            }
        } else {
            // 2-bit packed query, read through a cached 64-bit window
            uint32_t cw = 0xFFFFFFFFu, wlo = 0, whi = 0;
            auto field = [&](uint32_t sympos, uint32_t nbits) -> uint32_t {      // symbols [sympos, sympos + nbits/2)
                uint64_t bit = 2 * (off + sympos);
                uint32_t wi = (uint32_t)(bit >> 5);
                if (wi != cw) {
                    cw = wi;
                    wlo = __ldg(qpk + wi);
                    whi = __ldg(qpk + wi + 1);
                }
                uint32_t v = __funnelshift_r(wlo, whi, (uint32_t)bit & 31u);
                return nbits >= 32 ? v : (v & ((1u << nbits) - 1u));
            };
            uint32_t pos = L;
            if (o2.kmer_k && L >= o2.kmer_k) {
                // the first kmer_k symbols in one lookup
                uint2 e = __ldg(o2.kmer + field(L - o2.kmer_k, 2 * o2.kmer_k));
                lb = e.x;
                len = e.y;
                pos = L - o2.kmer_k;
                lines += 1;
            }
            while (pos > 0 && len > 0) {
                if (len == 1 && pos >= kTextCheckMin && o2.isa) {
                    // single row with pos symbols left: where the row sits in the text decides the rest (Occ2View::isa).  Every lane
                    // issues the same single lookups (one request each); each lane compares one 32-byte quarter of a text line.
                    const RowPos rp = row_pos<true>(o2.rowpos, lb, lines);
                    if (rp.pos < pos) { len = 0; break; }    // the read would start before its sequence
                    const uint32_t g0 = rp.g - pos;
                    lb = __ldg(o2.isa + g0);       // the final row, fetched together with the text lines (only kept on a match)
                    lines += 1;
                    if (out_at && sub == 3) out_at[q] = make_uint2(rp.seq, rp.pos - pos);      // replaced by kNoSeq below on a mismatch
                    // lane `sub` compares the read's words sub, sub + 4, ... (symbols [16 j, 16 j + 16)) with the text at g0 + 16 j: the
                    // group's four lanes read four consecutive text words per step, within one or two 128-byte lines
                    uint32_t bad = 0;
                    for (uint32_t j = sub; 16 * j < pos; j += 4) {
                        const uint32_t x = g0 + 16 * j, cnt = min(16u, pos - 16 * j);
                        const uint32_t t = __funnelshift_r(__ldg(o2.text32 + (x >> 4)), __ldg(o2.text32 + (x >> 4) + 1), 2 * (x & 15));
                        const uint32_t m = cnt >= 16 ? 0xFFFFFFFFu : (1u << (2 * cnt)) - 1u;
                        bad |= (t ^ field(16 * j, 32)) & m;
                    }
                    bad |= __shfl_xor_sync(gmask, bad, 1);
                    bad |= __shfl_xor_sync(gmask, bad, 2);
                    lines += ((g0 + pos - 1) >> 9) - (g0 >> 9) + 1;
                    if (bad) { len = 0; break; }
                    checked = true;
                    break;
                }
                if (len == 1 && pos >= 16 && o2.jump) {
                    // single-row interval: 16 symbols per lookup through the LF^16 jump table -- or 32 when the table holds the merged
                    // 16-byte entries and the next 32 symbols stay inside one sequence
                    uint2 e, f = make_uint2(kJumpInvalid, 0);
                    if (o2.jump_wide) {
                        const uint4 w = __ldg(reinterpret_cast<const uint4*>(o2.jump) + lb);
                        e = make_uint2(w.x, w.y);
                        f = make_uint2(w.z, w.w);
                    } else {
                        e = __ldg(o2.jump + lb);
                    }
                    lines += 1;
                    if (e.x != kJumpInvalid) {
                        if (e.y != field(pos - 16, 32)) { len = 0; break; }
                        if (pos >= 32 && f.x != kJumpInvalid) {
                            if (f.y != field(pos - 32, 32)) { len = 0; break; }
                            lb = f.x;
                            pos -= 32;
                            continue;
                        }
                        lb = e.x;
                        pos -= 16;
                        continue;
                    }
                }
                if (len == 1 && pos >= 4 && o2.jump4) {
                    // ... and four symbols per lookup through the LF^4 table for what is left of the pattern
                    uint2 e = __ldg(o2.jump4 + lb);
                    lines += 1;
                    if (e.x != kJumpInvalid) {
                        if (e.y != field(pos - 4, 8)) { len = 0; break; }
                        lb = e.x;
                        pos -= 4;
                        continue;
                    }
                }
                if (pos == 1) {
                    extend_left_uni(ix, lb, len, field(0, 2) + 1, dummy);
                    lines += 1;
                    break;
                }
                const uint32_t code = field(pos - 2, 4);          // (y-1)*4 + (x-1), x = query[pos-2], y = query[pos-1]
                const row_t hi = lb + len;
                const uint32_t b0 = lb >> 7, b1 = hi >> 7;
                Quarter q0 = load_quarter(o2, b0, sub);
                uint32_t p0, p1;
                if (b1 == b0) {
                    p0 = rank2_part(q0, sub, lb, code);
                    p1 = rank2_part(q0, sub, hi, code);
                    lines += 1;
                } else {
                    Quarter q1 = load_quarter(o2, b1, sub);
                    p0 = rank2_part(q0, sub, lb, code);
                    p1 = rank2_part(q1, sub, hi, code);
                    lines += 2;
                }
                uint32_t r0 = group_sum4(p0, gmask), r1 = group_sum4(p1, gmask);
                if (code == 0) {
                    r0 -= specials_below(o2, lb);
                    r1 -= specials_below(o2, hi);
                }
                lb = o2.C2[code] + r0;
                len = r1 - r0;
                pos -= 2;
            }
        }
        // the hit record of the query (dense: len == 0 when the pattern does not occur) + its length for locate's scan: the four
        // lanes of the group hold the same state, three of them write 8 bytes of the 24-byte record each (a warp's eight records are
        // 192 contiguous bytes), the fourth the length
        {
            uint2* rec = reinterpret_cast<uint2*>(out_hits + q);
            if (sub == 0) rec[0] = make_uint2(q + qidx_base, lb);           // qidx, lb
            else if (sub == 1) rec[1] = make_uint2(0u, len);                 // lb_rev, len
            else if (sub == 2) rec[2] = make_uint2(L, 0u);                   // steps, e
            else {
                out_len[q] = len;
                if (out_at && !checked) out_at[q] = make_uint2(kNoSeq, 0u);
            }
        }
        if (sub == 0) {
            found = len ? 1u : 0u;
            rows = len;
        }
    }
    // [2] = line requests issued by this kernel (physical work), counted once per group; [4] hits, [5] rows of all hits
    block_count3(counters, 2, sub == 0 ? lines : 0, 4, found, 5, rows);
}

// ---------------------------------------------------------------------------------------------------------
// K5: ordered compaction of the per-query intervals into hit records
// ---------------------------------------------------------------------------------------------------------
__global__ void flag_nonzero_kernel(const uint32_t* __restrict__ len, uint64_t count, uint32_t* __restrict__ flag) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    flag[i] = len[i] ? 1u : 0u;
}
__global__ void compact_exact_hits_kernel(const uint32_t* __restrict__ lb, const uint32_t* __restrict__ len,
                                          const uint32_t* __restrict__ pos, const uint64_t* __restrict__ qoff, uint32_t nq, uint32_t qidx_base,
                                          HitRec* __restrict__ hits) {
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    uint32_t l = len[q];
    if (!l) return;
    HitRec h;
    h.qidx = q + qidx_base; h.lb = lb[q]; h.lb_rev = 0; h.len = l;
    h.steps = (uint32_t)(qoff[q + 1] - qoff[q]);
    h.e = 0;
    hits[pos[q]] = h;
}
__global__ void hit_lengths_kernel(const HitRec* __restrict__ hits, uint64_t nh, uint32_t* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i > nh) return;
    out[i] = i < nh ? hits[i].len : 0;
}

// ---------------------------------------------------------------------------------------------------------
// K4: locate.  One SA row per thread; LF walk to the nearest sampled row (fmindex/BiFMIndex.h:177-202, walk_to_sample):
//     while row not sampled: c = BWT[row]; row = C[c] + rank(row, c); ++steps
// starts[] = exclusive prefix sum of the hit interval lengths; a thread finds its hit by binary search.
// ---------------------------------------------------------------------------------------------------------
// record of located row t: the largest h with starts[h] <= t (single: every record is exactly one row, h == t)
__device__ __forceinline__ uint32_t hit_of(const uint32_t* __restrict__ starts, uint32_t nh, uint32_t t, uint32_t single) {
    uint32_t lo = single ? t : 0, hi = single ? t + 1 : nh;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(starts + mid) <= t) lo = mid; else hi = mid;
    }
    return lo;
}
// the row of located row t in its record h
__device__ __forceinline__ row_t hit_row(const HitRec* __restrict__ hits, const uint32_t* __restrict__ starts, uint32_t h, uint32_t t, uint32_t single) {
    return __ldg(&hits[h].lb) + (single ? 0u : t - __ldg(starts + h));
}

template <class OCC>
__global__ void __launch_bounds__(256) locate_kernel(const __grid_constant__ IndexView<OCC> ix, const HitRec* __restrict__ hits,
                                                     const uint32_t* __restrict__ starts, uint32_t nh, uint32_t total, uint32_t single,
                                                     LocRec* __restrict__ out, unsigned long long* __restrict__ counters) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t steps = 0;
    if (t < total) {
        const uint32_t h = hit_of(starts, nh, t, single);
        const uint2 sample = __ldg(ix.samples + walk_to_sample(ix, hit_row(hits, starts, h, t, single), steps));
        LocRec r;
        r.qidx = __ldg(&hits[h].qidx); r.seq = sample.x; r.pos = sample.y + steps; r.e = __ldg(&hits[h].e);
        out[t] = r;
    }
    block_count2(counters, 2, steps, 1, steps);
}

// K4b: locate with the combined 64-byte locate blocks.  A pair of lanes owns one SA row: the even lane fetches the
// occ half of the block (symbol + rank -> next row), the odd lane the marker half (sampled? which sample?); two
// shuffles per LF step exchange "sampled" and the next row.  One line request per step instead of two.
__global__ void build_locblocks_kernel(const DnaBlock* __restrict__ occ, const uint4* __restrict__ marks, uint64_t nblocks, uint4* __restrict__ out) {
    uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const uint4* o = reinterpret_cast<const uint4*>(occ + b);
    uint4 m = marks[b];
    out[b * 4 + 0] = o[0];
    out[b * 4 + 1] = o[1];
    out[b * 4 + 2] = m;
    out[b * 4 + 3] = make_uint4(0, 0, 0, 0);
}

// one step of the pair walk: 1 + the sample index when `row` is sampled, else 0 and `row` becomes the next row (role 0 = occ half,
// role 1 = marker half; pmask = the pair's two lanes)
__device__ __forceinline__ uint32_t pair_step(const IndexView<OccDna>& ix, uint32_t role, uint32_t pmask, row_t& row) {
    uint32_t a0, a1, a2, a3, a4, a5, a6, a7;
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3), "=r"(a4), "=r"(a5), "=r"(a6), "=r"(a7)
                 : "l"(ix.locblocks + ((size_t)(row >> 6) * 4 + role * 2)));
    uint32_t mine;                                       // role 1: sampled ? 1 + sample index : 0;  role 0: next row
    if (role) {
        uint64_t bits = (uint64_t)a0 | ((uint64_t)a1 << 32);
        uint32_t o = row & 63;
        mine = ((bits >> o) & 1) ? 1u + a2 + __popcll(bits & low_mask(o)) : 0u;
    } else {
        DnaBlock b;
        b.cnt[0] = a0; b.cnt[1] = a1; b.cnt[2] = a2; b.cnt[3] = a3;
        b.p0 = (uint64_t)a4 | ((uint64_t)a5 << 32);
        b.p1 = (uint64_t)a6 | ((uint64_t)a7 << 32);
        const OccDna& occ = ix.occ[0];
        uint32_t c = occ.symbol(b, row);
        mine = ix.C[c] + occ.rank(b, row, c);
    }
    uint32_t other = __shfl_xor_sync(pmask, mine, 1);
    uint32_t sampled = role ? mine : other;
    if (!sampled) row = role ? other : mine;
    return sampled;
}

__global__ void __launch_bounds__(256) locate_pair_kernel(const __grid_constant__ IndexView<OccDna> ix, const HitRec* __restrict__ hits,
                                                          const uint32_t* __restrict__ starts, uint32_t nh, uint32_t total, uint32_t single,
                                                          LocRec* __restrict__ out, unsigned long long* __restrict__ counters) {
    // Persistent lane pairs with refill: LF walks take 0 .. rate-1 steps, so a warp of fixed rows idles half of its
    // lanes while the longest walk finishes.  Here a pair that reaches its sample immediately takes the next row
    // (t += number of pairs in the grid); all pairs run the same loop body, there is no divergence to pay for.
    const uint32_t npairs = (gridDim.x * blockDim.x) >> 1;
    uint32_t t = (blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    const uint32_t role = threadIdx.x & 1;
    const uint32_t pmask = 3u << (threadIdx.x & 30);
    uint32_t steps_total = 0, steps = 0;
    row_t row = 0;
    uint32_t qidx = 0, err = 0;
    auto fetch = [&]() {
        const uint32_t h = hit_of(starts, nh, t, single);
        row = hit_row(hits, starts, h, t, single);
        qidx = __ldg(&hits[h].qidx);
        err = __ldg(&hits[h].e);
        steps = 0;
    };
    bool active = t < total;
    if (active) fetch();
    while (active) {
        const uint32_t sampled = pair_step(ix, role, pmask, row);
        if (sampled) {
            if (role == 0) {
                uint2 sample = __ldg(ix.samples + (sampled - 1));
                LocRec r;
                r.qidx = qidx; r.seq = sample.x; r.pos = sample.y + steps; r.e = err;
                out[t] = r;
                steps_total += steps;
            }
            t += npairs;
            active = t < total;
            if (active) fetch();
        } else {
            ++steps;
        }
    }
    block_count2(counters, 2, steps_total, 1, steps_total);
}

// K4c: locate shortcut table.  locrow[row] = sample_index << step_bits | steps of the LF walk of `row` (built by walking every row
// once with the lane-pair walk above); locate(row) then is locrow[row] + samples[index]: two line fetches instead of ~10.
__global__ void __launch_bounds__(256) locrow_build_kernel(const __grid_constant__ IndexView<OccDna> ix, uint32_t step_bits, uint32_t* __restrict__ out,
                                                           uint32_t* __restrict__ overflow) {
    const uint64_t npairs = ((uint64_t)gridDim.x * blockDim.x) >> 1;
    uint64_t t = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    const uint32_t role = threadIdx.x & 1;
    const uint32_t pmask = 3u << (threadIdx.x & 30);
    uint32_t steps = 0;
    row_t row = (row_t)t;
    bool active = t < ix.n;
    while (active) {
        const uint32_t sampled = pair_step(ix, role, pmask, row);
        if (sampled) {
            if (role == 0) {
                const uint32_t idx = sampled - 1;
                if (steps >= (1u << step_bits) || idx >= (1u << (32 - step_bits))) atomicOr(overflow, 1u);
                out[t] = (idx << step_bits) | steps;
            }
            t += npairs;
            active = t < ix.n;
            row = (row_t)t;
            steps = 0;
        } else {
            ++steps;
        }
    }
}

// the same table for any layout: one thread per row walks to its sample with separate occ / marker loads (build time only)
template <class OCC>
__global__ void __launch_bounds__(256) locrow_build_gen_kernel(const __grid_constant__ IndexView<OCC> ix, uint32_t step_bits, uint32_t* __restrict__ out,
                                                               uint32_t* __restrict__ overflow) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ix.n) return;
    uint32_t steps = 0;
    const uint32_t idx = walk_to_sample(ix, (row_t)t, steps, 1u << 20);
    if (idx == kNoSample) { atomicOr(overflow, 1u); out[t] = 0; return; }     // no sample on this walk (cannot be located anyway)
    if (steps >= (1u << step_bits) || idx >= (1u << (32 - step_bits))) atomicOr(overflow, 1u);
    out[t] = (idx << step_bits) | steps;
}

// Text check tables (fmb_index::isa / text2), one thread per row: (seq, pos) of the row from the locate shortcut, g = start[seq] + pos;
// isa[g] = row, and BWT[row] is the symbol at g - 1 (a delimiter when pos == 0: those positions keep code 0, no read window reaches
// them).  flags[0] = a row outside its sequence, flags[1] = the largest LF step count of any row.
__global__ void __launch_bounds__(256) text_tables_kernel(const __grid_constant__ IndexView<OccDna> ix, const __grid_constant__ RowPosView rp,
                                                          const uint32_t* __restrict__ start, uint32_t nseq, uint32_t* __restrict__ isa,
                                                          uint32_t* __restrict__ text, uint32_t* __restrict__ flags) {
    const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    uint32_t steps = 0;
    if (r < ix.n) {
        uint32_t lines = 0;
        const RowPos p = row_pos<false>(rp, (row_t)r, lines);
        steps = p.steps;
        if (p.seq >= nseq || p.pos >= __ldg(start + p.seq + 1) - __ldg(start + p.seq)) {
            atomicOr(flags, 1u);
        } else {
            const uint32_t g = __ldg(start + p.seq) + p.pos;
            isa[g] = (uint32_t)r;
            if (p.pos) {
                const DnaBlock b = ix.occ[0].load((uint32_t)(r >> 6), 0);
                const uint32_t c = ix.occ[0].symbol(b, (row_t)r);
                atomicOr(text + ((g - 1) >> 4), ((c - 1) & 3u) << (2 * ((g - 1) & 15)));
            }
        }
    }
    steps = __reduce_max_sync(0xFFFFFFFFu, steps);
    if ((threadIdx.x & 31) == 0 && steps) atomicMax(flags + 1, steps);
}
// text-regular sampling at rate R = 1 + the largest step count: every sample at a multiple of R (then the step count of every row is
// pos % R: its sample is the one multiple of R in (pos - R, pos])
__global__ void __launch_bounds__(256) sample_rate_kernel(const uint2* __restrict__ samples, uint64_t count, uint32_t rate, uint32_t* __restrict__ bad) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < count && samples[i].y % rate) atomicOr(bad, 1u);
}
// the locate shortcut turned into the suffix array in place (text-regular sampling, after text_tables_kernel checked every row):
// rows[r] = g of row r, rows = rp.locrow (each thread reads its own word once, before it overwrites it)
__global__ void __launch_bounds__(256) sa_from_locrow_kernel(const __grid_constant__ RowPosView rp, uint64_t n, uint32_t* rows) {
    const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (r >= n) return;
    uint32_t lines = 0;
    rows[r] = row_pos<true>(rp, (row_t)r, lines).g;
}

// K4d: locate through the shortcut table in either form (RowPosView): the suffix array (one fetch per row plus the cached sequence
// entry; sampling is text-regular, so the walk would take pos % rate steps) or the shortcut word plus the sample.
// at (may be nullptr): (seq, pos) per record found by the text check of exact search (kNoSeq: not checked); with text-regular sampling
// at rate rp.rate such a row needs pos % rate LF steps and no index access
__global__ void __launch_bounds__(256) locate_shortcut_kernel(const __grid_constant__ RowPosView rp, const HitRec* __restrict__ hits,
                                                              const uint32_t* __restrict__ starts, uint32_t nh, uint32_t total, uint32_t single,
                                                              const uint2* __restrict__ at, LocRec* __restrict__ out,
                                                              unsigned long long* __restrict__ counters) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t steps = 0;
    if (t < total) {
        const uint32_t h = hit_of(starts, nh, t, single);
        LocRec r;
        r.qidx = __ldg(&hits[h].qidx); r.e = __ldg(&hits[h].e);
        const uint2 a = at ? __ldg(at + h) : make_uint2(kNoSeq, 0u);      // a checked hit is a single row
        if (a.x != kNoSeq) {
            steps = a.y % rp.rate;
            r.seq = a.x; r.pos = a.y;
        } else {
            uint32_t lines = 0;
            const RowPos p = row_pos<false>(rp, hit_row(hits, starts, h, t, single), lines);
            steps = p.steps;
            r.seq = p.seq; r.pos = p.pos;
        }
        out[t] = r;
    }
    // the LF steps the walk WOULD take: the algorithmic work of SURVEY.md §8d stays reported
    block_count2(counters, 2, steps, 1, steps);
}

// index.locate(row) for arbitrary rows (fmindex/BiFMIndex.h:177-202): same LF walk as locate_kernel, row list input
template <class OCC>
__global__ void __launch_bounds__(256) locate_rows_kernel(const __grid_constant__ IndexView<OCC> ix, const uint64_t* __restrict__ rows, uint64_t count,
                                                          uint32_t* __restrict__ seq, uint32_t* __restrict__ pos, uint64_t* __restrict__ steps_out) {
    uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= count) return;
    uint32_t steps = 0;
    const uint2 sample = __ldg(ix.samples + walk_to_sample(ix, (row_t)rows[t], steps));
    seq[t] = sample.x;
    pos[t] = sample.y;
    steps_out[t] = steps;
}

// Measurement aid (SURVEY.md §8d "empirical ceiling"): independent -- not pointer chasing -- random gathers over one of the index's
// own tables.  A group of LANES lanes fetches one aligned granule of PER * LANES bytes with ONE load instruction per lane, exactly
// like the search kernels do (4 x 32 B for a pair line, 1 x 16 B for a jump entry, 1 x 32 B for an occ block); the addresses come
// from a counter hash, so every load of a thread is independent of the ones before it.
template <int PER, int LANES>
__global__ void __launch_bounds__(256) gather_probe_kernel(const char* __restrict__ tab, uint64_t ngran, uint32_t iters, uint32_t* __restrict__ out) {
    const uint64_t tid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint64_t group = tid / LANES;
    const uint32_t lane = (uint32_t)(tid % LANES);
    uint32_t acc = 0;
#pragma unroll 4
    for (uint32_t i = 0; i < iters; ++i) {
        const uint64_t g = splitmix64(group * iters + i) % ngran;
        const char* p = tab + g * (uint64_t)(PER * LANES) + lane * PER;
        if (PER == 8) {
            const uint2 x = __ldg(reinterpret_cast<const uint2*>(p));
            acc ^= x.x ^ x.y;
        } else if (PER == 16) {
            const uint4 x = __ldg(reinterpret_cast<const uint4*>(p));
            acc ^= x.x ^ x.y ^ x.z ^ x.w;
        } else {
            uint32_t a, b, c, d, e, f, g2, h;
            asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(a), "=r"(b), "=r"(c), "=r"(d), "=r"(e), "=r"(f), "=r"(g2), "=r"(h) : "l"(p));
            acc ^= a ^ b ^ c ^ d ^ e ^ f ^ g2 ^ h;
        }
    }
    if (acc == 0x12345678u) out[0] = acc;      // keeps the loads alive
}

// annotatedArray.value(row) (suffixarray/SparseArray.h:63-70)
template <class OCC>
__global__ void sample_value_kernel(IndexView<OCC> ix, const uint64_t* __restrict__ rows, uint64_t count, uint8_t* __restrict__ has,
                                    uint32_t* __restrict__ seq, uint32_t* __restrict__ pos) {
    uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= count) return;
    row_t row = (row_t)rows[t];
    uint4 m = __ldg(ix.marks + (row >> 6));
    uint64_t bits = (uint64_t)m.x | ((uint64_t)m.y << 32);
    uint32_t o = row & 63;
    bool h = (bits >> o) & 1;
    has[t] = h ? 1 : 0;
    uint2 sample = make_uint2(0, 0);
    if (h) sample = __ldg(ix.samples + (m.z + __popcll(bits & low_mask(o))));
    seq[t] = sample.x;
    pos[t] = sample.y;
}

}  // namespace fmb
