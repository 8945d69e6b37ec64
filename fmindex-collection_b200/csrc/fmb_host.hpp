// fmb_host.hpp -- host-side objects behind the opaque handles of include/fmb200.h.
#pragma once
#include <cstdint>
#include <cstdio>
#include <mutex>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/fmb200.h"
#include "fmb_device.cuh"

namespace fmb {

void set_error(const char* fmt, ...);
void note_launches(unsigned n);   // bookkeeping for fmb_kernel_launch_count()

// Caching device allocator: cudaMalloc / cudaFree cost 0.1 - 1 ms each and cudaFree synchronises the device, which
// dominated a search step made of ~10 temporary buffers.  Freed blocks up to 16 GB (40 GB in total) are kept per device in size
// classes (<= 12.5 % internal waste) and handed out again; every API call synchronises its stream before it
// returns a block, so a cached block never has work pending.  pool_trim() gives everything back to CUDA.
void* pool_alloc(size_t bytes);   // nullptr + set_error on failure
void pool_free(void* p);
void pool_trim();

#define FMB_CUDA(call)                                                                               \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess) {                                                                     \
            fmb::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return e_ == cudaErrorMemoryAllocation ? FMB_ENOMEM : FMB_ECUDA;                         \
        }                                                                                            \
    } while (0)

#define FMB_TRY(expr)                  \
    do {                               \
        int rc_ = (expr);              \
        if (rc_ != FMB_OK) return rc_; \
    } while (0)

// device buffer with RAII
template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
        return *this;
    }
    ~DevBuf() { release(); }
    void release() {
        if (p) pool_free(p);
        p = nullptr;
        n = 0;
    }
    int alloc(size_t count) {
        release();
        if (count == 0) count = 1;
        p = static_cast<T*>(pool_alloc(count * sizeof(T)));
        if (!p) return FMB_ENOMEM;
        n = count;
        return FMB_OK;
    }
    size_t bytes() const { return n * sizeof(T); }
};

// internal record formats (compact, 32-bit: n < 2^32)
struct HitRec {
    uint32_t qidx, lb, lb_rev, len, steps, e;
};
typedef fmb_loc32 LocRec;
struct SmemRec {                  // fmb_smem with 32-bit fields
    uint32_t qidx, begin, end, lb, len;
};

}  // namespace fmb

struct fmb_index {
    int device = 0;
    int sm_count = 0;                    // SMs of `device` (launch geometry of the persistent kernels)
    uint32_t sigma = 0;
    uint64_t n = 0;
    bool bidirectional = false;
    bool dna = true;                     // 2-bit layout (sigma <= 5 with delimiter); else the generic layout
    uint32_t first_symb = 1;             // 0: BiFMIndex::NoDelim (symbol 0 is an ordinary symbol, omega-sorted text)
    bool reuse_rev = false;              // BiFMIndex::ReuseRev: the one BWT (of text + reversed text) serves both directions
    cudaStream_t stream = nullptr;       // stream all work of this index is enqueued on
    cudaStream_t own_stream = nullptr;   // private stream created with the index
    fmb::DevBuf<fmb::DnaBlock> occ_dna[2];
    fmb::DevBuf<uint8_t> occ_gen[2];
    uint32_t gen_stride = 0, gen_planes = 0;
    fmb::DevBuf<uint32_t> delim_rows[2];
    uint64_t n_delims = 0;
    uint32_t delim0[2] = {0, 0};
    fmb::DevBuf<uint4> marks;
    fmb::DevBuf<uint2> samples;
    fmb::DevBuf<uint4> locblocks;        // combined occ + marker records for locate (sigma <= 5)
    fmb::DevBuf<uint32_t> locrow;        // locate shortcut: per row sample index << loc_step_bits | LF steps
    uint32_t loc_step_bits = 0;
    int locate_mode = 0;                 // FMB_LOCATE_*
    uint64_t n_samples = 0;
    uint64_t C[65] = {0};
    // two-symbol table (OccDna2) of direction 0, sigma <= 5 only
    fmb::DevBuf<uint4> occ2;
    fmb::DevBuf<uint32_t> specials;
    uint32_t n_specials = 0;
    uint32_t special01[2] = {0xFFFFFFFFu, 0xFFFFFFFFu};
    uint32_t C2[16] = {};
    fmb::DevBuf<uint2> jump[2];          // LF^16 jump tables
    uint32_t jump_shift[2] = {0, 0};     // 1: the table holds 16-byte entries {LF^16, 16 symbols, LF^32, 16 more symbols} (two uint2 per row)
    fmb::DevBuf<uint2> jump4[2];         // LF^4 jump tables (same entry format, 4 symbols in the low 8 bits)
    fmb::DevBuf<uint2> kmer;             // k-mer interval table of direction 0
    uint32_t kmer_k = 0;
    fmb::DevBuf<uint4> bikmer;           // bidirectional k-mer table for scheme-search roots
    uint32_t bikmer_k = 0;
    int exact_mode = 0;                  // FMB_EXACT_*
    // text check of exact search (FMB_TEXT_CHECK, built from the locate shortcut): isa[g] = row of text position g of s0 0 s1 0 ...,
    // text2 = the text as 2-bit codes (symbol - 1), 16 per word, position g at bits 2 (g % 16) of word g / 16, and seq_start[s] = g of
    // the first symbol of sequence s (+ n at the end).  text_rate = R when a row is sampled iff its position is a multiple of R
    // (FMB_TEXT_LOCATE: the located row of a checked read needs pos % R LF steps), else 0.
    fmb::DevBuf<uint32_t> isa, text2, seq_start_d;
    uint32_t text_rate = 0;
    // suffix array (FMB_TABLE_LOCROW in place of `locrow` when text_rate is set on the DNA layout): sa[row] = g of the row's suffix,
    // one fetch per located row (the LF steps the walk would take are pos % text_rate); seq_of_block finds the sequence of a g
    // (fmb_device.cuh seq_of)
    fmb::DevBuf<uint32_t> sa;
    fmb::DevBuf<uint2> seq_of_block;
    // optional tables this image is allowed to hold (FMB_TABLE_* bits), decided once by plan_tables (csrc/fmb_lib.cu) from the image
    // budget (fmb_set_image_budget / FMB_IMAGE_GB; default: everything the device can hold) and the FMB_NO_* knobs of its knob table
    uint32_t allowed_tables = 0xFFFFFFFFu;
    // engine of the one-call end-to-end path (persistent worker threads + streams, csrc/fmb_engine.cu), created on first use
    mutable void* engine = nullptr;
    mutable std::mutex engine_mu;
    // text extraction (csrc/fmb_extract.cu), built on the first call that needs it under anchor_mu: per sequence its length, its
    // offset in the text s0 0 s1 0 ... and the row of its delimiter; then the anchor table -- text positions with known rows, sorted
    // by position (every sample plus every delimiter), as two parallel arrays
    mutable std::mutex anchor_mu;
    mutable bool layout_ready = false;
    mutable std::vector<uint64_t> seq_len, seq_start;
    mutable std::vector<uint32_t> seq_delim_row;
    mutable fmb::DevBuf<uint32_t> anchor_pos, anchor_row;
    mutable uint64_t n_anchors = 0;

    fmb::IndexView<fmb::OccDna> view_dna() const;
    fmb::IndexView<fmb::OccGen> view_gen() const;
    fmb::Occ2View view_occ2() const;
    fmb::RowPosView view_rowpos() const;   // the locate shortcut table in either form
    uint64_t device_bytes() const;

    // The image's device buffers, the one list that device_bytes() and fmb_index_replicate walk: f(buffer of a, the same buffer of
    // b, replicated).  The anchor table is counted in the image but not replicated: a replica builds its own on first use.
    template <class A, class B, class F>
    static void for_each_buffer(A& a, B& b, F&& f) {
        for (int d = 0; d < 2; ++d) {
            f(a.occ_dna[d], b.occ_dna[d], true);
            f(a.occ_gen[d], b.occ_gen[d], true);
            f(a.delim_rows[d], b.delim_rows[d], true);
            f(a.jump[d], b.jump[d], true);
            f(a.jump4[d], b.jump4[d], true);
        }
        f(a.occ2, b.occ2, true);
        f(a.specials, b.specials, true);
        f(a.marks, b.marks, true);
        f(a.samples, b.samples, true);
        f(a.locblocks, b.locblocks, true);
        f(a.locrow, b.locrow, true);
        f(a.kmer, b.kmer, true);
        f(a.bikmer, b.bikmer, true);
        f(a.isa, b.isa, true);
        f(a.text2, b.text2, true);
        f(a.seq_start_d, b.seq_start_d, true);
        f(a.sa, b.sa, true);
        f(a.seq_of_block, b.seq_of_block, true);
        f(a.anchor_pos, b.anchor_pos, false);
        f(a.anchor_row, b.anchor_row, false);
    }
};

namespace fmb {
// Stream the calling thread enqueues the work of `ix` on: a per-thread override (used by the pipelined
// search+locate path, where several host threads drive one index on their own streams) or the index's stream.
extern thread_local cudaStream_t tls_stream_override;
inline cudaStream_t active_stream(const fmb_index* ix) { return tls_stream_override ? tls_stream_override : ix->stream; }
void engine_destroy(fmb_index* ix);   // joins the worker threads of the index's engine, if it has one

// ---- index image construction (K1, csrc/fmb_lib.cu), shared by fmb_index_create_ex and fmb_index_build --------------------------
int use_device(int device);
int new_index(fmb_index** out, int device, uint32_t sigma, uint64_t n, bool bidirectional, uint32_t flags);
uint64_t image_budget();                                           // bytes, 0 = no limit
uint32_t plan_tables(const fmb_index* ix, uint64_t n_samples);     // the FMB_TABLE_* bits for ix->allowed_tables
constexpr uint32_t kTableTextCheck = 1u << 16;                     // allowed_tables bit of the text check tables (FMB_TEXT_CHECK)
constexpr uint32_t kTableSuffixArray = 1u << 17;                   // ... and of the suffix array in place of the locate shortcut
int ensure_layout(const fmb_index* ix);                            // sequence lengths and starts (csrc/fmb_extract.cu)
int build_occ_from_device_bwt(fmb_index* ix, int dir, const uint8_t* d_bwt);
int compute_C(fmb_index* ix);
// after compute_C: pair + k-mer tables (DNA layout), the LF jump tables of directions 0 and 1, the merged LF^32 entries and the
// bidirectional k-mer table
int build_search_tables(fmb_index* ix);
// after the marks: locate blocks (DNA layout), the locate shortcut, then the text check tables built from it
int build_locate_tables(fmb_index* ix);

inline unsigned grid_for(uint64_t items, unsigned block) {
    uint64_t g = (items + block - 1) / block;
    return (unsigned)(g ? g : 1);
}

struct EventTimer {           // device time between construction and stop() on stream s
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t s;
    explicit EventTimer(cudaStream_t s_) : s(s_) {
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, s);
    }
    double stop() {
        cudaEventRecord(b, s);
        cudaEventSynchronize(b);
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        return ms;
    }
    ~EventTimer() {
        cudaEventDestroy(a);
        cudaEventDestroy(b);
    }
};

// exclusive prefix sum of u32 -> u32 on `stream`, synchronised (CUB; plumbing, not a hot kernel)
int exclusive_sum_u32(const uint32_t* in, uint32_t* out, uint64_t count, cudaStream_t stream);
}  // namespace fmb

struct fmb_queries {
    int device = 0;
    uint64_t nq = 0;
    uint64_t qidx_base = 0;           // added to every reported qidx (chunked uploads)
    uint64_t total_symbols = 0;
    uint32_t max_len = 0, min_len = 0;
    uint64_t h2d_bytes = 0;           // bytes the upload copied host -> device
    fmb::DevBuf<uint8_t> symbols;     // padded to a multiple of 16 bytes
    fmb::DevBuf<uint64_t> offsets;    // nq + 1
    fmb::DevBuf<uint32_t> packed;     // sigma <= 5: 2-bit codes (symbol-1), 16 per word (+2 words of padding)
    fmb::DevBuf<uint8_t> flags;       // sigma <= 5: 1 = query holds a symbol without 2-bit code (0 or >= sigma)
};

struct fmb_results {
    int device = 0;
    int kind = 0;                     // 0 = hits, 1 = located rows, 2 = SMEMs, 3 = located rows of SMEMs
    uint64_t count = 0;               // hits (cursors with a non-empty interval) / located rows / SMEMs
    fmb::DevBuf<fmb::HitRec> hits;
    fmb::DevBuf<fmb::LocRec> locs;    // kind 3: qidx holds the number of the SMEM record the row belongs to
    fmb::DevBuf<fmb::SmemRec> smems;  // kinds 2 and 3 (csrc/fmb_smem.cu); kind 2 also fills `at` per record
    // exact search leaves its hits DENSE: one record per query (`slots` of them, len == 0 for queries without hit) plus the
    // interval lengths as a separate array -- locate works on that directly, the records are compacted only when they are fetched
    uint64_t slots = 0;               // records in `hits` (== count unless dense)
    bool dense = false;
    fmb::DevBuf<uint32_t> lens;       // dense results: len of every record (+ one trailing 0), the input of locate's scan
    fmb::DevBuf<uint2> at;            // dense exact results with the text check: (seq, pos) of every checked hit, kNoSeq elsewhere
                                      // (SMEMs: of every record the text path found)
    uint64_t total_rows = UINT64_MAX; // sum of the interval lengths when the search kernel counted it, else unknown
    fmb_stats stats{};
};
