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
    // two-symbol table (OccDna2), sigma <= 5 only
    fmb::DevBuf<uint4> occ2[2];
    fmb::DevBuf<uint32_t> specials[2];
    uint32_t n_specials[2] = {0, 0};
    uint32_t special01[2][2] = {{0xFFFFFFFFu, 0xFFFFFFFFu}, {0xFFFFFFFFu, 0xFFFFFFFFu}};
    uint32_t C2[2][16] = {};
    fmb::DevBuf<uint2> jump[2];          // LF^16 jump tables
    uint32_t jump_shift[2] = {0, 0};     // 1: the table holds 16-byte entries {LF^16, 16 symbols, LF^32, 16 more symbols} (two uint2 per row)
    fmb::DevBuf<uint2> jump4[2];         // LF^4 jump tables (same entry format, 4 symbols in the low 8 bits)
    fmb::DevBuf<uint2> kmer;             // k-mer interval table of direction 0
    uint32_t kmer_k = 0;
    fmb::DevBuf<uint4> bikmer;           // bidirectional k-mer table for scheme-search roots
    uint32_t bikmer_k = 0;
    int exact_mode = 0;                  // FMB_EXACT_*
    // optional tables this image is allowed to hold (FMB_TABLE_* bits), decided once from the image budget (fmb_set_image_budget /
    // FMB_IMAGE_GB; default: everything the device can hold)
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
    fmb::Occ2View view_occ2(int dir) const;
    uint64_t device_bytes() const;
};

namespace fmb {
// Stream the calling thread enqueues the work of `ix` on: a per-thread override (used by the pipelined
// search+locate path, where several host threads drive one index on their own streams) or the index's stream.
extern thread_local cudaStream_t tls_stream_override;
inline cudaStream_t active_stream(const fmb_index* ix) { return tls_stream_override ? tls_stream_override : ix->stream; }
void engine_destroy(fmb_index* ix);   // joins the worker threads of the index's engine, if it has one
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
    int kind = 0;                     // 0 = hits, 1 = located rows
    uint64_t count = 0;               // hits (cursors with a non-empty interval) / located rows
    fmb::DevBuf<fmb::HitRec> hits;
    fmb::DevBuf<fmb::LocRec> locs;
    // exact search leaves its hits DENSE: one record per query (`slots` of them, len == 0 for queries without hit) plus the
    // interval lengths as a separate array -- locate works on that directly, the records are compacted only when they are fetched
    uint64_t slots = 0;               // records in `hits` (== count unless dense)
    bool dense = false;
    fmb::DevBuf<uint32_t> lens;       // dense results: len of every record (+ one trailing 0), the input of locate's scan
    uint64_t total_rows = UINT64_MAX; // sum of the interval lengths when the search kernel counted it, else unknown
    fmb_stats stats{};
};
