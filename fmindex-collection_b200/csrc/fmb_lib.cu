// fmb_lib.cu -- index image construction (K1), String_c / cursor batch kernels, exact search (K2),
// locate (K4), result compaction (K5) and the C-ABI of include/fmb200.h.
#include <algorithm>
#include <cstdarg>
#include <cstring>
#include <atomic>
#include <map>
#include <mutex>
#include <unordered_map>

#include <cub/cub.cuh>

#include "fmb_host.hpp"
#include "fmb_kernels.cuh"

namespace fmb {

static thread_local std::string g_error = "";
thread_local cudaStream_t tls_stream_override = nullptr;
static std::atomic<uint64_t> g_launches{0};

void note_launches(unsigned n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
}

// ---- caching device allocator (see fmb_host.hpp) ------------------------------------------------------------
namespace {
struct Pool {
    std::mutex mu;
    std::multimap<std::pair<int, size_t>, void*> free_blocks;      // (device, class size) -> block
    std::unordered_map<void*, std::pair<int, size_t>> live;         // block -> (device, class size)
    size_t cached_bytes = 0;
};
Pool& pool() {
    static Pool* p = new Pool();     // intentionally leaked: must outlive static destructors that free buffers
    return *p;
}
constexpr size_t kMaxCachedBlock = size_t(1) << 34;      // blocks above 16 GB go straight back to CUDA
size_t size_class(size_t bytes) {
    if (bytes <= 4096) return 4096;
    // blocks that are never cached need no size class: 2 MB granularity instead of up to 12.5 % slack (3 GB per 24 GB jump table)
    if (bytes > kMaxCachedBlock) return (bytes + (size_t(2) << 20) - 1) / (size_t(2) << 20) * (size_t(2) << 20);
    int top = 63 - __builtin_clzll((unsigned long long)bytes);
    size_t step = size_t(1) << (top - 3);
    return (bytes + step - 1) / step * step;
}
constexpr size_t kMaxCachedTotal = size_t(40) << 30;     // ... and so does anything that would push the cache above 40 GB
}  // namespace

void pool_trim() {
    Pool& P = pool();
    std::lock_guard<std::mutex> lk(P.mu);
    for (auto& kv : P.free_blocks) cudaFree(kv.second);
    P.free_blocks.clear();
    P.cached_bytes = 0;
}

void* pool_alloc(size_t bytes) {
    Pool& P = pool();
    int dev = 0;
    cudaGetDevice(&dev);
    size_t cls = size_class(bytes);
    {
        std::lock_guard<std::mutex> lk(P.mu);
        auto it = P.free_blocks.find({dev, cls});
        if (it != P.free_blocks.end()) {
            void* p = it->second;
            P.free_blocks.erase(it);
            P.cached_bytes -= cls;
            P.live[p] = {dev, cls};
            return p;
        }
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, cls);
    if (e != cudaSuccess) {
        cudaGetLastError();
        pool_trim();
        e = cudaMalloc(&p, cls);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cudaMalloc(%zu bytes) failed: %s", cls, cudaGetErrorString(e));
        return nullptr;
    }
    std::lock_guard<std::mutex> lk(P.mu);
    P.live[p] = {dev, cls};
    return p;
}

void pool_free(void* p) {
    if (!p) return;
    Pool& P = pool();
    std::lock_guard<std::mutex> lk(P.mu);
    auto it = P.live.find(p);
    if (it == P.live.end()) { cudaFree(p); return; }
    auto key = it->second;
    P.live.erase(it);
    if (key.second > kMaxCachedBlock || P.cached_bytes + key.second > kMaxCachedTotal) { cudaFree(p); return; }
    P.free_blocks.insert({key, p});
    P.cached_bytes += key.second;
}

int use_device(int device) {
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess || cnt == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s); libfmb200 has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return FMB_ENODEVICE;
    }
    if (device < 0 || device >= cnt) {
        set_error("device %d out of range (have %d)", device, cnt);
        return FMB_ENODEVICE;
    }
    FMB_CUDA(cudaSetDevice(device));
    return FMB_OK;
}

// cudaMalloc for buffers handed to the caller (fmb_device_free); the allocator's cached blocks are given back first when memory is short
static int raw_alloc(uint8_t** p, size_t bytes) {
    cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        pool_trim();
        e = cudaMalloc(p, bytes);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? FMB_ENOMEM : FMB_ECUDA;
    }
    return FMB_OK;
}

int exclusive_sum_u32(const uint32_t* in, uint32_t* out, uint64_t count, cudaStream_t stream) {
    size_t tmp_bytes = 0;
    FMB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, in, out, (int64_t)count, stream));
    DevBuf<uint8_t> tmp;
    FMB_TRY(tmp.alloc(tmp_bytes));
    FMB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, in, out, (int64_t)count, stream));
    FMB_CUDA(cudaStreamSynchronize(stream));
    return FMB_OK;
}

// in-place exclusive scan of `count` values of a custom type with `op` on `stream`, not synchronised (CUB)
template <typename T, typename Op>
static int exclusive_scan(T* data, uint64_t count, Op op, T init, cudaStream_t stream) {
    size_t tmp_bytes = 0;
    FMB_CUDA(cub::DeviceScan::ExclusiveScan(nullptr, tmp_bytes, data, data, op, init, (int64_t)count, stream));
    DevBuf<uint8_t> tmp;
    FMB_TRY(tmp.alloc(tmp_bytes));
    FMB_CUDA(cub::DeviceScan::ExclusiveScan(tmp.p, tmp_bytes, data, data, op, init, (int64_t)count, stream));
    return FMB_OK;
}

struct ToU64 {
    __host__ __device__ unsigned long long operator()(uint32_t v) const { return v; }
};
struct Uint4Add {
    __host__ __device__ uint4 operator()(const uint4& a, const uint4& b) const {
        return make_uint4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    }
};

}  // namespace fmb

using namespace fmb;

fmb::IndexView<fmb::OccDna> fmb_index::view_dna() const {
    fmb::IndexView<fmb::OccDna> v{};
    for (int d = 0; d < 2; ++d) {
        const int src = reuse_rev ? 0 : d;          // ReuseRev: extendRight reads the same BWT (fmindex/BiFMIndexCursor.h fetchRightBwt)
        v.occ[d].blocks = occ_dna[src].p;
        v.occ[d].delim_rows = delim_rows[src].p;
        v.occ[d].n_delims = (uint32_t)n_delims;
        v.occ[d].delim0 = delim0[src];
    }
    for (uint32_t s = 0; s <= sigma; ++s) v.C[s] = (uint32_t)C[s];
    v.n = (row_t)n;
    v.sigma = sigma;
    v.first_symb = first_symb;
    v.marks = marks.p;
    v.samples = samples.p;
    v.locblocks = locblocks.p;
    return v;
}

fmb::IndexView<fmb::OccGen> fmb_index::view_gen() const {
    fmb::IndexView<fmb::OccGen> v{};
    for (int d = 0; d < 2; ++d) {
        v.occ[d].blocks = occ_gen[reuse_rev ? 0 : d].p;
        v.occ[d].stride = gen_stride;
        v.occ[d].planes = gen_planes;
        v.occ[d].sigma = sigma;
    }
    for (uint32_t s = 0; s <= sigma; ++s) v.C[s] = (uint32_t)C[s];
    v.n = (row_t)n;
    v.sigma = sigma;
    v.first_symb = first_symb;
    v.marks = marks.p;
    v.samples = samples.p;
    v.locblocks = nullptr;
    return v;
}

// run `...` with V bound to the device view of the index's layout (kernels deduce OCC from it)
#define FMB_DISPATCH(ix, V, ...)                    \
    do {                                            \
        if ((ix)->dna) {                            \
            auto V = (ix)->view_dna();              \
            __VA_ARGS__;                            \
        } else {                                    \
            auto V = (ix)->view_gen();              \
            __VA_ARGS__;                            \
        }                                           \
    } while (0)

fmb::Occ2View fmb_index::view_occ2() const {
    fmb::Occ2View v{};
    v.lines = occ2.p;
    v.specials = specials.p;
    v.n_specials = n_specials;
    v.s0 = special01[0];
    v.s1 = special01[1];
    for (int i = 0; i < 16; ++i) v.C2[i] = C2[i];
    v.jump = jump[0].p;
    v.jump_wide = jump_shift[0];
    v.jump4 = jump4[0].p;
    v.kmer = kmer.p;
    v.kmer_k = kmer_k;
    v.isa = isa.p;
    v.text32 = text2.p;
    v.rowpos = view_rowpos();
    return v;
}

fmb::RowPosView fmb_index::view_rowpos() const {
    return fmb::RowPosView{sa.p, seq_of_block.p, seq_start_d.p, locrow.p, samples.p, loc_step_bits, text_rate};
}

uint64_t fmb_index::device_bytes() const {
    uint64_t b = 0;
    for_each_buffer(*this, *this, [&](const auto& buf, const auto&, bool) { b += buf.bytes(); });
    return b;
}

// ---------------------------------------------------------------------------------------------------------
// index construction from BWT bytes that are already on the device
// ---------------------------------------------------------------------------------------------------------
namespace fmb {

// ---- image budget: which accelerating tables an index may hold ----------------------------------------------------------------
// Every table beyond the occurrence blocks is optional (results never depend on them); they trade HBM for speed.  With a budget
// the tables are admitted in the order of what they buy per byte (measured: profiles/r02_image_budget_curve.json):
//   pair table + k-mer table (exact search: two symbols per line, the first 14 symbols in one lookup), locate blocks,
//   LF^16 table of direction 0 (sixteen symbols per lookup once an interval is a single row), LF^16 of direction 1 (text windows of
//   the k-error searches in both directions), bidirectional k-mer table, locate shortcut, merged LF^32 entries, LF^4 tables, text check
//   tables (ISA + 2-bit text: exact-search reads decided on the text; last because they serve exact search alone).
// DNA layout, both k-mer tables: largest k <= 14 with 8 * 4^k <= n (the exact-search table, 8 bytes per k-mer, stays below ~n bytes)
static uint32_t dna_kmer_k(uint64_t n) {
    uint32_t k = 0;
    while (k < 14 && (uint64_t(8) << (2 * (k + 1))) <= n) ++k;
    return k;
}
// generic layout: largest k <= 8 whose table of (sigma - first_symb)^k entries stays below 2 n bytes (1 Gaa, sigma = 21: k = 6, 1 GB)
static uint32_t gen_bikmer_k(const fmb_index* ix) {
    const uint64_t base = ix->sigma - ix->first_symb;
    uint32_t k = 0;
    uint64_t count = 1;
    while (k < 8 && base > 1 && count * base * 16 <= 2 * ix->n && count * base < (uint64_t(1) << 31)) { count *= base; ++k; }
    return k;
}
static std::atomic<uint64_t> g_image_budget{0};          // bytes, 0 = no limit
uint64_t image_budget() {
    uint64_t b = g_image_budget.load();
    if (!b) {
        static const double env_gb = getenv("FMB_IMAGE_GB") ? atof(getenv("FMB_IMAGE_GB")) : 0.0;
        if (env_gb > 0) b = (uint64_t)(env_gb * 1e9);
    }
    return b;
}
static uint32_t budget_tables(const fmb_index* ix, uint64_t n_samples) {
    const uint64_t budget = image_budget();
    if (!budget) return 0xFFFFFFFFu;
    const double n = (double)ix->n;
    // what is always there: occurrence blocks (both directions), marks + samples
    double used = (ix->dna ? n / 2 : n / 64 * 128) * (ix->bidirectional && !ix->reuse_rev ? 2 : 1) + n / 4 + 8.0 * (double)n_samples;
    uint32_t allowed = 0;
    auto admit = [&](uint32_t bits, double bytes) {
        if (used + bytes <= (double)budget) { used += bytes; allowed |= bits; return true; }
        return false;
    };
    if (ix->dna) {
        const uint32_t k = dna_kmer_k(ix->n);
        admit(FMB_TABLE_PAIR | FMB_TABLE_KMER, n + 8.0 * (double)(uint64_t(1) << (2 * k)));
        admit(FMB_TABLE_LOCBLOCK, n);
        const bool j0 = admit(FMB_TABLE_JUMP, 8 * n);
        const bool j1 = ix->bidirectional && admit(FMB_TABLE_JUMP_REV, 8 * n);
        if (ix->bidirectional) admit(FMB_TABLE_BIKMER, 16.0 * (double)(uint64_t(1) << (2 * k)));
        if (allowed & FMB_TABLE_LOCBLOCK) admit(FMB_TABLE_LOCROW, 4 * n);
        if (j0) admit(FMB_TABLE_JUMP32, 8 * n);
        if (j0) admit(FMB_TABLE_JUMP4, 8 * n * (j1 ? 2 : 1));
        if (allowed & FMB_TABLE_LOCROW) admit(kTableTextCheck | kTableSuffixArray, 4.25 * n + n / 512);      // + the sequence lookup of sa
    } else {
        admit(FMB_TABLE_JUMP4, 8 * n * (ix->bidirectional ? 2 : 1));      // generic layout: byte-symbol LF^4 tables ...
        admit(FMB_TABLE_LOCROW, 4 * n);                                    // ... the locate shortcut ...
        if (ix->bidirectional) {                                           // ... and the bidirectional k-mer table of the scheme roots
            double cnt = 1;
            for (uint32_t p = 0; p < gen_bikmer_k(ix); ++p) cnt *= (double)(ix->sigma - ix->first_symb);
            admit(FMB_TABLE_BIKMER, 16 * cnt);
        }
    }
    return allowed;
}

// The tables admitted by the budget, less those of the knobs set in the environment, read on every build.  The knobs are applied
// after admission, so a knob frees no budget for later tables.  Knob table:
//   knob               DNA layout (sigma <= 5 with delimiter) clears   generic layout clears
//   FMB_NO_JUMP        JUMP, JUMP_REV, JUMP4, JUMP32                    JUMP4 (its only jump tables)
//   FMB_NO_JUMP32      JUMP32                                           -
//   FMB_NO_JUMP4       JUMP4                                            -
//   FMB_NO_BIKMER      BIKMER                                           BIKMER
//   FMB_NO_LOCBLOCKS   LOCBLOCK, LOCROW (the shortcut walks the blocks) -
//   FMB_NO_LOCROW      LOCROW                                           LOCROW
//   FMB_NO_TEXTCHECK   the text check tables (kTableTextCheck)          -
//   FMB_NO_SA          the suffix array (kTableSuffixArray): LOCROW     -
//                      keeps the form sample index + steps
// (the text check tables are built from the locate shortcut: without LOCROW there are none; the suffix array replaces the shortcut
// when the text check finds the sampling text-regular)
// FMB_KMER_K (build_occ2) sizes the exact-search k-mer table; FMB_KMER_K=0 leaves it out.
uint32_t plan_tables(const fmb_index* ix, uint64_t n_samples) {
    static const struct { const char* name; uint32_t dna, gen; } knobs[] = {
        {"FMB_NO_JUMP", FMB_TABLE_JUMP | FMB_TABLE_JUMP_REV | FMB_TABLE_JUMP4 | FMB_TABLE_JUMP32, FMB_TABLE_JUMP4},
        {"FMB_NO_JUMP32", FMB_TABLE_JUMP32, 0},
        {"FMB_NO_JUMP4", FMB_TABLE_JUMP4, 0},
        {"FMB_NO_BIKMER", FMB_TABLE_BIKMER, FMB_TABLE_BIKMER},
        {"FMB_NO_LOCBLOCKS", FMB_TABLE_LOCBLOCK | FMB_TABLE_LOCROW, 0},
        {"FMB_NO_LOCROW", FMB_TABLE_LOCROW, FMB_TABLE_LOCROW},
        {"FMB_NO_TEXTCHECK", kTableTextCheck, 0},
        {"FMB_NO_SA", kTableSuffixArray, 0},
    };
    uint32_t allowed = budget_tables(ix, n_samples);
    for (const auto& k : knobs)
        if (getenv(k.name)) allowed &= ~(ix->dna ? k.dna : k.gen);
    return allowed;
}

// Builds occ table `dir` of `ix` from n BWT bytes at d_bwt (device).  Fails when a symbol is >= sigma.
int build_occ_from_device_bwt(fmb_index* ix, int dir, const uint8_t* d_bwt) {
    const uint64_t n = ix->n;
    const uint64_t nblocks = n / 64 + 1;
    cudaStream_t st = active_stream(ix);
    if (!ix->dna) {
        // generic layout: planes + exclusive prefix counts per 64 rows (fmb_device.cuh OccGen)
        uint32_t planes = 1;
        while ((1u << planes) < ix->sigma) ++planes;
        ix->gen_planes = planes;
        ix->gen_stride = (8 * planes + 4 * (ix->sigma - 1) + 31) / 32 * 32;
        FMB_TRY(ix->occ_gen[dir].alloc(nblocks * ix->gen_stride + 64));
        FMB_CUDA(cudaMemsetAsync(ix->occ_gen[dir].p, 0, nblocks * ix->gen_stride + 64, st));
        DevBuf<Cnt32> counts;
        FMB_TRY(counts.alloc(nblocks));
        DevBuf<uint32_t> bad;
        FMB_TRY(bad.alloc(1));
        FMB_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(uint32_t), st));
        pack_gen_kernel<<<grid_for(nblocks, 128), 128, 0, st>>>(d_bwt, n, ix->sigma, planes, ix->gen_stride, ix->occ_gen[dir].p, counts.p, bad.p);
        FMB_CUDA(cudaGetLastError());
        uint32_t h_bad = 0;
        FMB_CUDA(cudaMemcpyAsync(&h_bad, bad.p, sizeof h_bad, cudaMemcpyDeviceToHost, st));
        FMB_CUDA(cudaStreamSynchronize(st));
        if (h_bad) { set_error("BWT contains a symbol >= sigma (%u)", ix->sigma); return FMB_EINVAL; }
        // number of delimiter rows = total count of symbol 0 (last block's scanned count + its local count): take it from C later
        FMB_TRY(exclusive_scan(counts.p, nblocks, Cnt32Add{}, Cnt32{}, st));
        store_gen_counts_kernel<<<grid_for(nblocks, 128), 128, 0, st>>>(ix->occ_gen[dir].p, ix->gen_stride, planes, ix->sigma, counts.p, nblocks);
        FMB_CUDA(cudaGetLastError());
        FMB_CUDA(cudaStreamSynchronize(st));
        return FMB_OK;
    }
    FMB_TRY(ix->occ_dna[dir].alloc(nblocks));
    DevBuf<uint4> counts;
    FMB_TRY(counts.alloc(nblocks));
    DevBuf<uint32_t> dflags;     // per block: number of delimiter rows, then scanned
    FMB_TRY(dflags.alloc(nblocks + 1));
    DevBuf<uint32_t> bad;
    FMB_TRY(bad.alloc(1));
    FMB_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(uint32_t), st));
    pack_dna_kernel<<<grid_for(nblocks + 1, 256), 256, 0, st>>>(d_bwt, n, ix->sigma, ix->occ_dna[dir].p, counts.p, dflags.p, bad.p);
    FMB_CUDA(cudaGetLastError());
    uint32_t h_bad = 0;
    FMB_CUDA(cudaMemcpyAsync(&h_bad, bad.p, sizeof h_bad, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    if (h_bad) {
        set_error("BWT contains a symbol >= sigma (%u)", ix->sigma);
        return FMB_EINVAL;
    }
    FMB_TRY(exclusive_scan(counts.p, nblocks, Uint4Add{}, make_uint4(0, 0, 0, 0), st));      // per-block symbol counts
    store_counts_kernel<<<grid_for(nblocks, 256), 256, 0, st>>>(ix->occ_dna[dir].p, counts.p, nblocks);
    FMB_CUDA(cudaGetLastError());
    // delimiter rows: scan per-block delimiter counts, then scatter the rows
    FMB_TRY(exclusive_sum_u32(dflags.p, dflags.p, nblocks + 1, st));
    uint32_t nd = 0;
    FMB_CUDA(cudaMemcpy(&nd, dflags.p + nblocks, sizeof nd, cudaMemcpyDeviceToHost));
    if (dir == 0) ix->n_delims = nd;
    else if (ix->n_delims != nd) {
        set_error("bwt and bwtRev hold a different number of delimiters (%llu vs %u)", (unsigned long long)ix->n_delims, nd);
        return FMB_EINVAL;
    }
    FMB_TRY(ix->delim_rows[dir].alloc((size_t)nd + 1));
    FMB_CUDA(cudaMemsetAsync(ix->delim_rows[dir].p, 0xFF, ((size_t)nd + 1) * sizeof(uint32_t), st));
    if (nd) {
        scatter_delims_kernel<<<grid_for(nblocks, 256), 256, 0, st>>>(d_bwt, n, dflags.p, ix->delim_rows[dir].p);
        FMB_CUDA(cudaGetLastError());
    }
    FMB_CUDA(cudaMemcpyAsync(&ix->delim0[dir], ix->delim_rows[dir].p, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    return FMB_OK;
}

// C[s] = prefix_rank(n, s), s = 0..sigma (utils.h:200-206), evaluated with the device table itself
int compute_C(fmb_index* ix) {
    DevBuf<uint64_t> d_out;
    FMB_TRY(d_out.alloc(ix->sigma + 1));
    FMB_DISPATCH(ix, v, compute_C_kernel<<<1, 64, 0, ix->stream>>>(v, d_out.p));
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaMemcpyAsync(ix->C, d_out.p, (ix->sigma + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->stream));
    FMB_CUDA(cudaStreamSynchronize(ix->stream));
    if (!ix->dna) ix->n_delims = ix->C[1];          // rows holding symbol 0
    return FMB_OK;
}

// C2[code] = first row of the interval of the pattern "x y" = C[x] + rank(C[y], x), code = (y-1)*4 + (x-1)
__global__ void compute_C2_kernel(IndexView<OccDna> ix, int dir, uint32_t* out) {
    uint32_t code = threadIdx.x;
    if (code >= 16) return;
    uint32_t y = (code >> 2) + 1, x = (code & 3) + 1;
    const OccDna& occ = ix.occ[dir];
    row_t at = ix.C[y];
    DnaBlock b = occ.load(at >> 6);
    out[code] = (x < ix.sigma && y < ix.sigma) ? ix.C[x] + occ.rank(b, at, x) : 0u;
}

// bidirectional k-mer table (16 bytes per k-mer, k from dna_kmer_k / gen_bikmer_k); needs both occ tables and C
static int build_bikmer(fmb_index* ix) {
    if (!ix->bidirectional || !(ix->allowed_tables & FMB_TABLE_BIKMER)) return FMB_OK;
    if (!ix->dna) {
        const uint32_t k = gen_bikmer_k(ix), base = ix->sigma - ix->first_symb;
        if (k < 2) return FMB_OK;
        uint64_t count = 1;
        for (uint32_t p = 0; p < k; ++p) count *= base;
        cudaStream_t st = active_stream(ix);
        FMB_TRY(ix->bikmer.alloc(count));
        bikmer_table_gen_kernel<<<grid_for(count, 256), 256, 0, st>>>(ix->view_gen(), k, base, count, ix->bikmer.p);
        FMB_CUDA(cudaGetLastError());
        FMB_CUDA(cudaStreamSynchronize(st));
        note_launches(1);
        ix->bikmer_k = k;
        return FMB_OK;
    }
    const uint32_t k = dna_kmer_k(ix->n);
    if (k < 2) return FMB_OK;
    const uint64_t count = uint64_t(1) << (2 * k);
    cudaStream_t st = active_stream(ix);
    FMB_TRY(ix->bikmer.alloc(count));
    bikmer_table_kernel<<<grid_for(count, 256), 256, 0, st>>>(ix->view_dna(), k, count, ix->bikmer.p);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaStreamSynchronize(st));
    ix->bikmer_k = k;
    return FMB_OK;
}

// combined 64-byte locate records of the DNA layout (needs occ table 0 and the marks)
static int build_locblocks(fmb_index* ix) {
    if (!ix->marks.p || ix->n_samples == 0 || !(ix->allowed_tables & FMB_TABLE_LOCBLOCK)) return FMB_OK;
    const uint64_t nblocks = ix->n / 64 + 1;
    cudaStream_t st = active_stream(ix);
    FMB_TRY(ix->locblocks.alloc(nblocks * 4));
    build_locblocks_kernel<<<grid_for(nblocks, 256), 256, 0, st>>>(ix->occ_dna[0].p, ix->marks.p, nblocks, ix->locblocks.p);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaStreamSynchronize(st));
    return FMB_OK;
}

// locate shortcut table: walk every row once.  The word packs sample index and step count; when they do not fit 32 bits (very sparse
// or irregular sampling), or some walk never reaches a sample, the table is dropped and locate keeps walking.  On the DNA layout the
// walk reads the locate blocks: plan_tables allows LOCROW only together with LOCBLOCK, so build_locblocks has built them.
static int build_locrow(fmb_index* ix) {
    if (!ix->marks.p || ix->n_samples == 0 || !(ix->allowed_tables & FMB_TABLE_LOCROW)) return FMB_OK;
    uint32_t idx_bits = 1;
    while (idx_bits < 32 && (uint64_t(1) << idx_bits) < ix->n_samples) ++idx_bits;
    const uint32_t step_bits = 32 - idx_bits;
    size_t free_b = 0, total_b = 0;
    pool_trim();
    FMB_CUDA(cudaMemGetInfo(&free_b, &total_b));
    if (step_bits < 1 || (double)free_b <= 4.0 * (double)ix->n * 1.5 + (double)(1u << 28)) return FMB_OK;
    cudaStream_t st = active_stream(ix);
    FMB_TRY(ix->locrow.alloc(ix->n));
    DevBuf<uint32_t> ovf;
    FMB_TRY(ovf.alloc(1));
    FMB_CUDA(cudaMemsetAsync(ovf.p, 0, sizeof(uint32_t), st));
    ix->loc_step_bits = step_bits;
    if (ix->dna) {               // persistent grid
        const unsigned grid = (unsigned)std::min<uint64_t>(grid_for(ix->n * 2, 256), (uint64_t)ix->sm_count * 8);
        locrow_build_kernel<<<grid, 256, 0, st>>>(ix->view_dna(), step_bits, ix->locrow.p, ovf.p);
    } else {                     // one thread per row
        locrow_build_gen_kernel<<<grid_for(ix->n, 256), 256, 0, st>>>(ix->view_gen(), step_bits, ix->locrow.p, ovf.p);
        note_launches(1);
    }
    FMB_CUDA(cudaGetLastError());
    uint32_t h_ovf = 0;
    FMB_CUDA(cudaMemcpyAsync(&h_ovf, ovf.p, sizeof h_ovf, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    if (h_ovf) {
        ix->locrow.release();
        ix->loc_step_bits = 0;
    }
    return FMB_OK;
}

// Builds the two-symbol table and the k-mer table of direction 0 from the one-symbol table (needs C).  sigma <= 5 only.
static int build_occ2(fmb_index* ix) {
    if (!(ix->allowed_tables & FMB_TABLE_PAIR)) return FMB_OK;
    const uint64_t n = ix->n;
    const uint64_t nblocks = n / 128 + 1, nquarters = nblocks * 4;
    cudaStream_t st = active_stream(ix);
    auto v = ix->view_dna();
    DevBuf<uint8_t> codes;
    FMB_TRY(codes.alloc(n));
    pair_codes_kernel<<<grid_for(n, 256), 256, 0, st>>>(v, 0, codes.p);
    FMB_CUDA(cudaGetLastError());
    FMB_TRY(ix->occ2.alloc(nblocks * 8));
    DevBuf<uint32_t> qcounts, scount;
    DevBuf<Cnt16> bcounts;
    FMB_TRY(qcounts.alloc(nquarters * 16));
    FMB_TRY(scount.alloc(nquarters + 1));
    FMB_TRY(bcounts.alloc(nblocks));
    pack_pairs_kernel<<<grid_for(nquarters + 1, 256), 256, 0, st>>>(codes.p, n, nblocks, ix->occ2.p, qcounts.p, scount.p);
    FMB_CUDA(cudaGetLastError());
    block_counts_kernel<<<grid_for(nblocks * 16, 256), 256, 0, st>>>(qcounts.p, nblocks, bcounts.p);
    FMB_CUDA(cudaGetLastError());
    FMB_TRY(exclusive_scan(bcounts.p, nblocks, Cnt16Add{}, Cnt16{}, st));
    store_pair_counts_kernel<<<grid_for(nquarters, 256), 256, 0, st>>>(ix->occ2.p, bcounts.p, nblocks);
    FMB_CUDA(cudaGetLastError());
    FMB_TRY(exclusive_sum_u32(scount.p, scount.p, nquarters + 1, st));
    uint32_t ns = 0;
    FMB_CUDA(cudaMemcpy(&ns, scount.p + nquarters, sizeof ns, cudaMemcpyDeviceToHost));
    FMB_TRY(ix->specials.alloc((size_t)ns + 2));
    FMB_CUDA(cudaMemsetAsync(ix->specials.p, 0xFF, ((size_t)ns + 2) * sizeof(uint32_t), st));
    if (ns) {
        scatter_specials_kernel<<<grid_for(nquarters, 256), 256, 0, st>>>(codes.p, n, nquarters, scount.p, ix->specials.p);
        FMB_CUDA(cudaGetLastError());
    }
    ix->n_specials = ns;
    FMB_CUDA(cudaMemcpyAsync(ix->special01, ix->specials.p, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    DevBuf<uint32_t> c2;
    FMB_TRY(c2.alloc(16));
    compute_C2_kernel<<<1, 32, 0, st>>>(v, 0, c2.p);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaMemcpyAsync(ix->C2, c2.p, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    uint32_t k = dna_kmer_k(n);                          // k-mer table
    const char* env = getenv("FMB_KMER_K");
    if (env) k = (uint32_t)std::min<long>(14, std::max<long>(0, atol(env)));
    ix->kmer_k = 0;
    if (k >= 2) {
        const uint64_t count = uint64_t(1) << (2 * k);
        FMB_TRY(ix->kmer.alloc(count));
        kmer_table_kernel<<<grid_for(count, 256), 256, 0, st>>>(v, k, count, ix->kmer.p);
        FMB_CUDA(cudaGetLastError());
        FMB_CUDA(cudaStreamSynchronize(st));
        ix->kmer_k = k;
    }
    return FMB_OK;
}

// LF^16 jump table of direction `dir` (8 bytes per row) by four rounds of pointer doubling.  Skipped -- the search then
// keeps taking two-symbol steps -- when the device cannot hold the two build buffers, or when the plan does not allow it.
static int build_jump(fmb_index* ix, int dir) {
    if (ix->dna ? !(ix->allowed_tables & (dir ? FMB_TABLE_JUMP_REV : FMB_TABLE_JUMP)) : !(ix->allowed_tables & FMB_TABLE_JUMP4)) return FMB_OK;
    const uint64_t n = ix->n;
    size_t free_b = 0, total_b = 0;
    pool_trim();
    FMB_CUDA(cudaMemGetInfo(&free_b, &total_b));
    if ((double)free_b < 2.0 * 8.0 * (double)n * 1.25 + (double)(1u << 28)) return FMB_OK;
    cudaStream_t st = active_stream(ix);
    DevBuf<uint2> a, b;
    FMB_TRY(a.alloc(n));
    FMB_TRY(b.alloc(n));
    if (!ix->dna) {
        // generic layout: LF^4 with the four symbols as bytes (two doubling rounds); compared with the raw query bytes
        jump_init_kernel<<<grid_for(n, 256), 256, 0, st>>>(ix->view_gen(), dir, a.p);
        FMB_CUDA(cudaGetLastError());
        for (uint32_t shift = 8; shift <= 16; shift *= 2) {
            jump_double_kernel<<<grid_for(n, 256), 256, 0, st>>>(a.p, b.p, n, shift, dir);
            FMB_CUDA(cudaGetLastError());
            std::swap(a, b);
        }
        FMB_CUDA(cudaStreamSynchronize(st));
        ix->jump4[dir] = std::move(a);
        return FMB_OK;
    }
    jump_init_kernel<<<grid_for(n, 256), 256, 0, st>>>(ix->view_dna(), dir, a.p);
    FMB_CUDA(cudaGetLastError());
    // LF^4 entries (after the second round) are kept as well when memory allows: they serve the tails shorter than 16 symbols
    const bool want4 = (ix->allowed_tables & FMB_TABLE_JUMP4) && (double)free_b > 3.0 * 8.0 * (double)n * 1.25 + (double)(size_t(24) << 30);
    for (uint32_t shift = 2; shift <= 16; shift *= 2) {
        // direction 0 is compared with query symbols to the LEFT of the match (farthest symbol = lowest position = low bits),
        // direction 1 with symbols to the RIGHT (nearest symbol = lowest position = low bits): both equal the packed query order
        jump_double_kernel<<<grid_for(n, 256), 256, 0, st>>>(a.p, b.p, n, shift, dir);
        FMB_CUDA(cudaGetLastError());
        std::swap(a, b);
        if (shift == 4 && want4) {
            FMB_TRY(ix->jump4[dir].alloc(n));
            FMB_CUDA(cudaMemcpyAsync(ix->jump4[dir].p, a.p, n * sizeof(uint2), cudaMemcpyDeviceToDevice, st));
        }
    }
    FMB_CUDA(cudaStreamSynchronize(st));
    ix->jump[dir] = std::move(a);
    return FMB_OK;
}

// Merged LF^16 / LF^32 table of direction 0 (16 bytes per row instead of 8): exact search then covers 32 symbols of a single-row
// interval per lookup.  Built after both LF^16 tables exist; skipped (the 8-byte table stays) when the device cannot hold the wide
// copy next to the narrow one plus what the remaining tables need, or when the plan does not allow it.
static int widen_jump0(fmb_index* ix) {
    if (!ix->dna || !ix->jump[0].p || ix->jump_shift[0] || !(ix->allowed_tables & FMB_TABLE_JUMP32)) return FMB_OK;
    const uint64_t n = ix->n;
    size_t free_b = 0, total_b = 0;
    pool_trim();
    FMB_CUDA(cudaMemGetInfo(&free_b, &total_b));
    // the wide table (16 n) next to the narrow one; the 8 n released afterwards cover the tables still to come (locate shortcut 4 n,
    // locate blocks n, marks, samples, bidirectional k-mer table)
    if ((double)free_b < 16.0 * (double)n * 1.125 + (double)(size_t(2) << 30)) return FMB_OK;
    cudaStream_t st = active_stream(ix);
    DevBuf<uint2> wide;
    FMB_TRY(wide.alloc(2 * n));
    jump_widen_kernel<<<grid_for(n, 256), 256, 0, st>>>(ix->jump[0].p, reinterpret_cast<uint4*>(wide.p), n);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaStreamSynchronize(st));
    note_launches(1);
    ix->jump[0] = std::move(wide);
    ix->jump_shift[0] = 1;
    pool_trim();
    return FMB_OK;
}

int build_search_tables(fmb_index* ix) {
    if (ix->dna) FMB_TRY(build_occ2(ix));
    FMB_TRY(build_jump(ix, 0));
    if (ix->bidirectional) FMB_TRY(build_jump(ix, 1));
    FMB_TRY(widen_jump0(ix));
    return build_bikmer(ix);
}

// Text check tables of exact search (DNA layout): ISA (4 bytes per row), the text as 2-bit codes and the sequence starts, built from
// the locate shortcut (every row's text position).  Skipped without the shortcut, when the plan does not allow them, when the device
// cannot hold them or when the samples do not describe a collection (the search then keeps its LF jumps).  text_rate is set when the
// sampling is text-regular, the condition under which locate can report the step counts of the rows the check finds; the locate
// shortcut then becomes the suffix array (kTableSuffixArray, knob FMB_NO_SA).
static int build_text_check(fmb_index* ix) {
    if (!ix->dna || !ix->locrow.p || !(ix->allowed_tables & kTableTextCheck)) return FMB_OK;
    const uint64_t n = ix->n, words = (n / 512 + 2) * 32;       // whole 128-byte lines and one more
    size_t free_b = 0, total_b = 0;
    pool_trim();
    FMB_CUDA(cudaMemGetInfo(&free_b, &total_b));
    if ((double)free_b <= 4.25 * (double)n * 1.1 + (double)(size_t(1) << 30)) return FMB_OK;
    if (ensure_layout(ix) != FMB_OK) return FMB_OK;
    const uint64_t nseq = ix->seq_start.size();
    std::vector<uint32_t> h_start(nseq + 1);
    for (uint64_t s = 0; s < nseq; ++s) h_start[s] = (uint32_t)ix->seq_start[s];
    h_start[nseq] = (uint32_t)n;
    cudaStream_t st = active_stream(ix);
    DevBuf<uint32_t> start, isa, text, flags;
    FMB_TRY(start.alloc(nseq + 1));
    FMB_TRY(isa.alloc(n));
    FMB_TRY(text.alloc(words));
    FMB_TRY(flags.alloc(3));
    FMB_CUDA(cudaMemcpyAsync(start.p, h_start.data(), (nseq + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    FMB_CUDA(cudaMemsetAsync(text.p, 0, words * sizeof(uint32_t), st));
    FMB_CUDA(cudaMemsetAsync(flags.p, 0, 3 * sizeof(uint32_t), st));
    text_tables_kernel<<<grid_for(n, 256), 256, 0, st>>>(ix->view_dna(), ix->view_rowpos(), start.p, (uint32_t)nseq, isa.p, text.p, flags.p);
    FMB_CUDA(cudaGetLastError());
    uint32_t h_flags[3] = {0, 0, 0};
    FMB_CUDA(cudaMemcpyAsync(h_flags, flags.p, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    if (h_flags[0]) return FMB_OK;
    const uint32_t rate = h_flags[1] + 1;
    sample_rate_kernel<<<grid_for(ix->n_samples, 256), 256, 0, st>>>(ix->samples.p, ix->n_samples, rate, flags.p + 2);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaMemcpyAsync(h_flags + 2, flags.p + 2, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    note_launches(2);
    ix->isa = std::move(isa);
    ix->text2 = std::move(text);
    ix->seq_start_d = std::move(start);
    ix->text_rate = h_flags[2] ? 0u : rate;
    // text-regular sampling: every row's step count is pos % text_rate, so the shortcut's sample index and steps say no more than the
    // row's text position -- the suffix array takes its place (same 4 bytes per row) and locates a row with one fetch
    if (ix->text_rate && (ix->allowed_tables & kTableSuffixArray) && nseq < (uint64_t(1) << 31)) {
        const uint64_t nb = (n >> 12) + 2;          // every block of a position < n, and the one after the last
        std::vector<uint2> sob(nb);
        uint64_t s = 0;
        for (uint64_t b = 0; b < nb; ++b) {
            const uint64_t first = b << 12;
            while (s + 1 < nseq && h_start[s + 1] <= first) ++s;
            const bool inner = s + 1 < nseq && h_start[s + 1] < first + 4096;
            sob[b] = make_uint2((uint32_t)s | (inner ? 1u << 31 : 0u), h_start[s]);
        }
        DevBuf<uint2> d_sob;
        FMB_TRY(d_sob.alloc(nb));
        FMB_CUDA(cudaMemcpyAsync(d_sob.p, sob.data(), nb * sizeof(uint2), cudaMemcpyHostToDevice, st));
        sa_from_locrow_kernel<<<grid_for(n, 256), 256, 0, st>>>(ix->view_rowpos(), n, ix->locrow.p);
        FMB_CUDA(cudaGetLastError());
        FMB_CUDA(cudaStreamSynchronize(st));
        note_launches(1);
        ix->sa = std::move(ix->locrow);
        ix->loc_step_bits = 0;
        ix->seq_of_block = std::move(d_sob);
    }
    return FMB_OK;
}

int build_locate_tables(fmb_index* ix) {
    if (ix->dna) FMB_TRY(build_locblocks(ix));
    FMB_TRY(build_locrow(ix));
    return build_text_check(ix);
}

// sample tables from a device bitmap ((n+63)/64 words; rows >= n clear) and device sample arrays
int build_marks_from_device(fmb_index* ix, const uint64_t* d_bitmap, const uint32_t* d_seq, const uint32_t* d_pos, uint64_t n_samples) {
    const uint64_t words = ix->n / 64 + 1;
    const uint64_t have = (ix->n + 63) / 64;
    cudaStream_t st = active_stream(ix);
    DevBuf<uint32_t> pc;
    FMB_TRY(pc.alloc(words + 1));
    popcount_words_kernel<<<grid_for(words + 1, 256), 256, 0, st>>>(d_bitmap, have, words + 1, pc.p);
    FMB_CUDA(cudaGetLastError());
    FMB_TRY(exclusive_sum_u32(pc.p, pc.p, words + 1, st));
    uint32_t total = 0;
    FMB_CUDA(cudaMemcpy(&total, pc.p + words, sizeof total, cudaMemcpyDeviceToHost));
    if (total != n_samples) {
        set_error("sample bitmap has %u set bits but n_samples = %llu", total, (unsigned long long)n_samples);
        return FMB_EINVAL;
    }
    FMB_TRY(ix->marks.alloc(words));
    build_marks_kernel<<<grid_for(words, 256), 256, 0, st>>>(d_bitmap, have, words, pc.p, ix->marks.p);
    FMB_CUDA(cudaGetLastError());
    FMB_TRY(ix->samples.alloc(n_samples));
    if (n_samples) {
        zip_samples_kernel<<<grid_for(n_samples, 256), 256, 0, st>>>(d_seq, d_pos, n_samples, ix->samples.p);
        FMB_CUDA(cudaGetLastError());
    }
    ix->n_samples = n_samples;
    FMB_CUDA(cudaStreamSynchronize(st));
    return FMB_OK;
}

int new_index(fmb_index** out, int device, uint32_t sigma, uint64_t n, bool bidirectional, uint32_t flags) {
    if (!out) { set_error("out is NULL"); return FMB_EINVAL; }
    *out = nullptr;
    if (sigma < 2 || sigma > 32) { set_error("sigma %u outside [2,32]", sigma); return FMB_EINVAL; }
    if (n == 0) { set_error("empty index"); return FMB_EINVAL; }
    if (n >= 0xFFFFFFFFull - 64) { set_error("n = %llu: this build supports n < 2^32 - 64", (unsigned long long)n); return FMB_EUNSUPPORTED; }
    FMB_TRY(use_device(device));
    fmb_index* ix = new fmb_index();
    ix->device = device;
    ix->sigma = sigma;
    ix->n = n;
    ix->bidirectional = bidirectional;
    ix->first_symb = (flags & FMB_INDEX_NO_DELIM) ? 0u : 1u;
    ix->reuse_rev = (flags & FMB_INDEX_REUSE_REV) != 0;
    // without delimiter symbol 0 is as frequent as any other symbol: the generic layout treats all symbols alike
    ix->dna = sigma <= 5 && ix->first_symb == 1;
    cudaError_t e = cudaStreamCreateWithFlags(&ix->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { set_error("cudaStreamCreate: %s", cudaGetErrorString(e)); delete ix; return FMB_ECUDA; }
    ix->stream = ix->own_stream;
    cudaDeviceGetAttribute(&ix->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (ix->sm_count < 1) ix->sm_count = 1;
    *out = ix;
    return FMB_OK;
}

template <typename T>
static int replicate_buf(DevBuf<T>& dst, const DevBuf<T>& src, int dst_dev, int src_dev, cudaStream_t st) {
    if (!src.p) return FMB_OK;
    FMB_TRY(dst.alloc(src.n));
    FMB_CUDA(cudaMemcpyPeerAsync(dst.p, dst_dev, src.p, src_dev, src.bytes(), st));
    return FMB_OK;
}

template <typename T>
static int upload(DevBuf<T>& buf, const T* host, size_t count, cudaStream_t st) {
    FMB_TRY(buf.alloc(count));
    if (count) FMB_CUDA(cudaMemcpyAsync(buf.p, host, count * sizeof(T), cudaMemcpyHostToDevice, st));
    return FMB_OK;
}

}  // namespace fmb

// =========================================================================================================
// C-ABI
// =========================================================================================================
extern "C" {

const char* fmb_last_error(void) { return fmb::g_error.c_str(); }
const char* fmb_version(void) { return "fmb200 0.1 (sm_100a)"; }

int fmb_device_count(void) {
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess) { cudaGetLastError(); return 0; }
    return cnt;
}

int fmb_index_create(fmb_index** out, int device, uint32_t sigma, uint64_t n, const uint8_t* bwt, const uint8_t* bwt_rev,
                     const uint64_t* sample_bitmap, const uint32_t* sample_seq, const uint32_t* sample_pos, uint64_t n_samples) {
    return fmb_index_create_ex(out, device, sigma, n, bwt, bwt_rev, sample_bitmap, sample_seq, sample_pos, n_samples, 0);
}

int fmb_index_create_ex(fmb_index** out, int device, uint32_t sigma, uint64_t n, const uint8_t* bwt, const uint8_t* bwt_rev,
                        const uint64_t* sample_bitmap, const uint32_t* sample_seq, const uint32_t* sample_pos, uint64_t n_samples, uint32_t flags) {
    if (!bwt) { set_error("bwt is NULL"); return FMB_EINVAL; }
    if (n_samples && (!sample_bitmap || !sample_seq || !sample_pos)) { set_error("sample arrays missing"); return FMB_EINVAL; }
    if (flags & ~(FMB_INDEX_NO_DELIM | FMB_INDEX_REUSE_REV)) { set_error("unknown index flags 0x%x", flags); return FMB_EINVAL; }
    if ((flags & FMB_INDEX_REUSE_REV) && bwt_rev) { set_error("a ReuseRev index has no bwtRev"); return FMB_EINVAL; }
    fmb_index* ix = nullptr;
    FMB_TRY(new_index(&ix, device, sigma, n, bwt_rev != nullptr || (flags & FMB_INDEX_REUSE_REV), flags));
    ix->allowed_tables = plan_tables(ix, n_samples);
    auto fail = [&](int rc) { fmb_index_destroy(ix); return rc; };
    {
        DevBuf<uint8_t> d_bwt;
        int rc = upload(d_bwt, bwt, n, ix->stream);
        if (rc) return fail(rc);
        rc = build_occ_from_device_bwt(ix, 0, d_bwt.p);
        if (rc) return fail(rc);
        if (bwt_rev) {
            cudaError_t e = cudaMemcpyAsync(d_bwt.p, bwt_rev, n, cudaMemcpyHostToDevice, ix->stream);
            if (e != cudaSuccess) { set_error("H2D bwtRev: %s", cudaGetErrorString(e)); return fail(FMB_ECUDA); }
            rc = build_occ_from_device_bwt(ix, 1, d_bwt.p);
            if (rc) return fail(rc);
        }
    }
    int rc = compute_C(ix);
    if (rc) return fail(rc);
    rc = build_search_tables(ix);
    if (rc) return fail(rc);
    {
        const uint64_t have = (n + 63) / 64;
        DevBuf<uint64_t> d_bm;
        DevBuf<uint32_t> d_seq, d_pos;
        std::vector<uint64_t> zero;
        if (!sample_bitmap) { zero.assign(have, 0); sample_bitmap = zero.data(); }
        rc = upload(d_bm, sample_bitmap, have, ix->stream);
        if (rc) return fail(rc);
        rc = upload(d_seq, sample_seq, n_samples, ix->stream);
        if (rc) return fail(rc);
        rc = upload(d_pos, sample_pos, n_samples, ix->stream);
        if (rc) return fail(rc);
        rc = build_marks_from_device(ix, d_bm.p, d_seq.p, d_pos.p, n_samples);
        if (rc) return fail(rc);
    }
    rc = build_locate_tables(ix);
    if (rc) return fail(rc);
    *out = ix;
    pool_trim();
    return FMB_OK;
}

// Copies the finished device image to another GPU (peer-to-peer when the two devices allow it; cudaMemcpyPeer stages through the
// host otherwise): a replica costs one pass over the image instead of another build.
int fmb_index_replicate(const fmb_index* src, int device, fmb_index** out) {
    if (!src || !out) { set_error("NULL argument"); return FMB_EINVAL; }
    *out = nullptr;
    if (device == src->device) { set_error("replica on the device of the original (%d)", device); return FMB_EINVAL; }
    fmb_index* ix = nullptr;
    FMB_TRY(new_index(&ix, device, src->sigma, src->n, src->bidirectional,
                      (src->first_symb ? 0u : FMB_INDEX_NO_DELIM) | (src->reuse_rev ? FMB_INDEX_REUSE_REV : 0u)));      // makes `device` current
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, device, src->device) == cudaSuccess && can) {
        cudaError_t pe = cudaDeviceEnablePeerAccess(src->device, 0);
        if (pe != cudaSuccess) cudaGetLastError();                                  // already enabled, or not possible: the copies still work
    }
    cudaGetLastError();
    auto fail = [&](int rc) { fmb_index_destroy(ix); return rc; };
    cudaStream_t st = ix->stream;
    // the source image must be complete before it is read
    {
        cudaError_t se = cudaSetDevice(src->device);
        if (se == cudaSuccess) se = cudaStreamSynchronize(src->stream);
        if (se == cudaSuccess) se = cudaSetDevice(device);
        if (se != cudaSuccess) { set_error("fmb_index_replicate: %s", cudaGetErrorString(se)); return fail(FMB_ECUDA); }
    }
    int rc = FMB_OK;
    fmb_index::for_each_buffer(*ix, *src, [&](auto& to, const auto& from, bool replicated) {
        if (!rc && replicated) rc = replicate_buf(to, from, device, src->device, st);
    });
    if (rc) return fail(rc);
    for (int d = 0; d < 2; ++d) {
        ix->delim0[d] = src->delim0[d];
        ix->jump_shift[d] = src->jump_shift[d];
    }
    ix->n_specials = src->n_specials;
    for (int i = 0; i < 2; ++i) ix->special01[i] = src->special01[i];
    for (int i = 0; i < 16; ++i) ix->C2[i] = src->C2[i];
    ix->gen_stride = src->gen_stride; ix->gen_planes = src->gen_planes;
    ix->n_delims = src->n_delims; ix->n_samples = src->n_samples;
    ix->loc_step_bits = src->loc_step_bits; ix->locate_mode = src->locate_mode; ix->exact_mode = src->exact_mode;
    ix->text_rate = src->text_rate;
    ix->kmer_k = src->kmer_k; ix->bikmer_k = src->bikmer_k;
    for (uint32_t s = 0; s <= src->sigma; ++s) ix->C[s] = src->C[s];
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { set_error("fmb_index_replicate: %s", cudaGetErrorString(e)); return fail(FMB_ECUDA); }
    *out = ix;
    return FMB_OK;
}

void fmb_index_destroy(fmb_index* ix) {
    if (!ix) return;
    engine_destroy(ix);
    cudaSetDevice(ix->device);
    if (ix->own_stream) cudaStreamDestroy(ix->own_stream);
    delete ix;
    pool_trim();
}

int fmb_index_get_info(const fmb_index* ix, fmb_index_info* info) {
    if (!ix || !info) { set_error("NULL argument"); return FMB_EINVAL; }
    std::lock_guard<std::mutex> lk(ix->anchor_mu);     // the anchor table may be being built by another thread
    memset(info, 0, sizeof *info);
    info->n = ix->n;
    info->sigma = ix->sigma;
    info->bidirectional = ix->bidirectional;
    info->n_samples = ix->n_samples;
    info->n_delims = ix->n_delims;
    info->device_bytes = ix->device_bytes();
    info->occ_block_bytes = ix->dna ? 32 : ix->gen_stride;
    info->occ_block_rows = 64;
    info->device = ix->device;
    info->flags = (ix->first_symb ? 0u : FMB_INDEX_NO_DELIM) | (ix->reuse_rev ? FMB_INDEX_REUSE_REV : 0u);
    info->tables = (ix->occ2.p ? FMB_TABLE_PAIR : 0) | (ix->kmer.p ? FMB_TABLE_KMER : 0) | (ix->jump[0].p ? FMB_TABLE_JUMP : 0) |
                   (ix->jump[1].p ? FMB_TABLE_JUMP_REV : 0) | (ix->locblocks.p ? FMB_TABLE_LOCBLOCK : 0) | (ix->locrow.p || ix->sa.p ? FMB_TABLE_LOCROW : 0) |
                   (ix->bikmer.p ? FMB_TABLE_BIKMER : 0) | (ix->jump4[0].p ? FMB_TABLE_JUMP4 : 0) | (ix->jump_shift[0] ? FMB_TABLE_JUMP32 : 0);
    info->tables |= ix->anchor_pos.p ? FMB_TABLE_ANCHORS : 0;
    info->text_tables = (ix->isa.p ? FMB_TEXT_CHECK : 0u) | (ix->isa.p && ix->text_rate ? FMB_TEXT_LOCATE : 0u);
    return FMB_OK;
}

int fmb_index_get_C(const fmb_index* ix, uint64_t* C) {
    if (!ix || !C) { set_error("NULL argument"); return FMB_EINVAL; }
    for (uint32_t s = 0; s <= ix->sigma; ++s) C[s] = ix->C[s];
    return FMB_OK;
}

int fmb_index_export(const fmb_index* ix, uint8_t* bwt, uint8_t* bwt_rev, uint64_t* sample_bitmap, uint32_t* sample_seq, uint32_t* sample_pos) {
    if (!ix) { set_error("NULL index"); return FMB_EINVAL; }
    FMB_TRY(use_device(ix->device));
    cudaStream_t st = active_stream(ix);
    for (int d = 0; d < 2; ++d) {
        uint8_t* dst = d ? bwt_rev : bwt;
        if (!dst) continue;
        if (d == 1 && (!ix->bidirectional || ix->reuse_rev)) { set_error("index has no bwtRev"); return FMB_EINVAL; }
        DevBuf<uint8_t> tmp;
        FMB_TRY(tmp.alloc(ix->n));
        FMB_DISPATCH(ix, v, unpack_bwt_kernel<<<grid_for(ix->n, 256), 256, 0, st>>>(v, d, tmp.p));
        FMB_CUDA(cudaGetLastError());
        FMB_CUDA(cudaMemcpyAsync(dst, tmp.p, ix->n, cudaMemcpyDeviceToHost, st));
        FMB_CUDA(cudaStreamSynchronize(st));
    }
    if (sample_bitmap) {
        const uint64_t have = (ix->n + 63) / 64;
        DevBuf<uint64_t> tmp;
        FMB_TRY(tmp.alloc(have));
        export_marks_kernel<<<grid_for(have, 256), 256, 0, st>>>(ix->marks.p, have, tmp.p);
        FMB_CUDA(cudaGetLastError());
        FMB_CUDA(cudaMemcpyAsync(sample_bitmap, tmp.p, have * 8, cudaMemcpyDeviceToHost, st));
        FMB_CUDA(cudaStreamSynchronize(st));
    }
    if ((sample_seq || sample_pos) && ix->n_samples) {
        std::vector<uint2> h(ix->n_samples);
        FMB_CUDA(cudaMemcpy(h.data(), ix->samples.p, ix->n_samples * sizeof(uint2), cudaMemcpyDeviceToHost));
        for (uint64_t i = 0; i < ix->n_samples; ++i) {
            if (sample_seq) sample_seq[i] = h[i].x;
            if (sample_pos) sample_pos[i] = h[i].y;
        }
    }
    return FMB_OK;
}

// raw bytes of the one-symbol occurrence table of direction `dir` (the blocks the kernels read): layout parity with fmb200::HostMirror
int fmb_index_export_blocks(const fmb_index* ix, int dir, uint8_t* out, uint64_t capacity, uint64_t* bytes, uint32_t* block_bytes) {
    if (!ix || !bytes) { set_error("NULL argument"); return FMB_EINVAL; }
    if (dir < 0 || dir > 1 || (dir == 1 && !ix->bidirectional)) { set_error("dir %d not available", dir); return FMB_EINVAL; }
    if (ix->reuse_rev) dir = 0;
    const uint64_t nblocks = ix->n / 64 + 1;
    const uint32_t stride = ix->dna ? 32u : ix->gen_stride;
    *bytes = nblocks * stride;
    if (block_bytes) *block_bytes = stride;
    if (!out) return FMB_OK;
    if (capacity < *bytes) { set_error("capacity %llu < %llu bytes", (unsigned long long)capacity, (unsigned long long)*bytes); return FMB_EOVERFLOW; }
    FMB_TRY(use_device(ix->device));
    const void* src = ix->dna ? (const void*)ix->occ_dna[dir].p : (const void*)ix->occ_gen[dir].p;
    FMB_CUDA(cudaStreamSynchronize(active_stream(ix)));
    FMB_CUDA(cudaMemcpy(out, src, *bytes, cudaMemcpyDeviceToHost));
    return FMB_OK;
}

// ---- String_c batch ops -----------------------------------------------------------------------------------
static int string_op(const fmb_index* ix, int dir, int op, const uint64_t* idx, const uint8_t* symb, uint64_t count,
                     uint64_t* out64, uint8_t* out8, uint64_t* out_prs) {
    if (!ix || !idx) { set_error("NULL argument"); return FMB_EINVAL; }
    if (dir < 0 || dir > 1 || (dir == 1 && !ix->bidirectional)) { set_error("dir %d not available", dir); return FMB_EINVAL; }
    FMB_TRY(use_device(ix->device));
    if (count == 0) return FMB_OK;
    for (uint64_t i = 0; i < count; ++i) {
        uint64_t lim = (op == 0) ? ix->n - 1 : ix->n;
        if (idx[i] > lim) { set_error("idx[%llu] = %llu out of range", (unsigned long long)i, (unsigned long long)idx[i]); return FMB_EINVAL; }
        if (symb && ((op == 2) ? symb[i] > ix->sigma : symb[i] >= ix->sigma)) { set_error("symbol %u out of range", symb[i]); return FMB_EINVAL; }
    }
    cudaStream_t st = active_stream(ix);
    DevBuf<uint64_t> d_idx, d_out, d_out2;
    DevBuf<uint8_t> d_symb;
    FMB_TRY(upload(d_idx, idx, count, st));
    if (symb) FMB_TRY(upload(d_symb, symb, count, st));
    size_t per = (op == 3) ? ix->sigma : 1;
    FMB_TRY(d_out.alloc(count * per));
    if (op == 3) FMB_TRY(d_out2.alloc(count * per));
    FMB_DISPATCH(ix, v, string_op_kernel<<<grid_for(count, 128), 128, 0, st>>>(v, dir, op, d_idx.p, d_symb.p, count, d_out.p, d_out2.p));
    FMB_CUDA(cudaGetLastError());
    std::vector<uint64_t> h(count * per);
    FMB_CUDA(cudaMemcpyAsync(h.data(), d_out.p, h.size() * 8, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    if (out8) for (uint64_t i = 0; i < count; ++i) out8[i] = (uint8_t)h[i];
    if (out64) memcpy(out64, h.data(), h.size() * 8);
    if (op == 3 && out_prs) FMB_CUDA(cudaMemcpy(out_prs, d_out2.p, h.size() * 8, cudaMemcpyDeviceToHost));
    return FMB_OK;
}

int fmb_string_symbol(const fmb_index* ix, int dir, const uint64_t* idx, uint64_t count, uint8_t* out) {
    return string_op(ix, dir, 0, idx, nullptr, count, nullptr, out, nullptr);
}
int fmb_string_rank(const fmb_index* ix, int dir, const uint64_t* idx, const uint8_t* symb, uint64_t count, uint64_t* out) {
    if (!symb) { set_error("symb is NULL"); return FMB_EINVAL; }
    return string_op(ix, dir, 1, idx, symb, count, out, nullptr, nullptr);
}
int fmb_string_prefix_rank(const fmb_index* ix, int dir, const uint64_t* idx, const uint8_t* symb, uint64_t count, uint64_t* out) {
    if (!symb) { set_error("symb is NULL"); return FMB_EINVAL; }
    return string_op(ix, dir, 2, idx, symb, count, out, nullptr, nullptr);
}
int fmb_string_all_ranks(const fmb_index* ix, int dir, const uint64_t* idx, uint64_t count, uint64_t* out_rs, uint64_t* out_prs) {
    return string_op(ix, dir, 3, idx, nullptr, count, out_rs, nullptr, out_prs);
}

// ---- cursor batch ops ---------------------------------------------------------------------------------------
static int cursor_op(const fmb_index* ix, int right, const uint64_t* cur, const uint8_t* symb, uint64_t count, uint64_t* out, bool all) {
    if (!ix || !cur || !out) { set_error("NULL argument"); return FMB_EINVAL; }
    if (!ix->bidirectional) { set_error("cursor ops need a bidirectional index"); return FMB_EINVAL; }
    FMB_TRY(use_device(ix->device));
    if (count == 0) return FMB_OK;
    for (uint64_t i = 0; i < count; ++i) {
        if (cur[4 * i] + cur[4 * i + 2] > ix->n || cur[4 * i + 1] + cur[4 * i + 2] > ix->n) { set_error("cursor %llu out of range", (unsigned long long)i); return FMB_EINVAL; }
        if (!all && symb[i] >= ix->sigma) { set_error("symbol out of range"); return FMB_EINVAL; }
    }
    cudaStream_t st = active_stream(ix);
    DevBuf<uint64_t> d_cur, d_out;
    DevBuf<uint8_t> d_symb;
    FMB_TRY(upload(d_cur, cur, count * 4, st));
    if (!all) FMB_TRY(upload(d_symb, symb, count, st));
    size_t per = all ? ix->sigma : 1;
    FMB_TRY(d_out.alloc(count * per * 4));
    FMB_DISPATCH(ix, v, cursor_op_kernel<<<grid_for(count, 128), 128, 0, st>>>(v, right, all ? 1 : 0, d_cur.p, d_symb.p, count, d_out.p));
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaMemcpyAsync(out, d_out.p, count * per * 4 * 8, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    return FMB_OK;
}
int fmb_cursor_extend(const fmb_index* ix, int right, const uint64_t* cur, const uint8_t* symb, uint64_t count, uint64_t* out) {
    if (!symb) { set_error("symb is NULL"); return FMB_EINVAL; }
    return cursor_op(ix, right, cur, symb, count, out, false);
}
int fmb_cursor_extend_all(const fmb_index* ix, int right, const uint64_t* cur, uint64_t count, uint64_t* out) {
    return cursor_op(ix, right, cur, nullptr, count, out, true);
}

// ---- queries ------------------------------------------------------------------------------------------------
// complement == nullptr: the batch as given; else reverse-complement doubling on the device (2 nq queries, only nq cross PCIe)
struct PackedInput {                      // 2-bit packed host symbols of the whole batch + exceptions (fmb_queries_upload_packed)
    const uint32_t* words = nullptr;
    const uint64_t* exc_pos = nullptr;
    const uint8_t* exc_sym = nullptr;
    uint64_t n_exc = 0;
};
static int upload_queries(fmb_queries** out, const fmb_index* ix, const uint8_t* symbols, const uint64_t* offsets, uint64_t nq, const uint8_t* complement,
                          const PackedInput* pk = nullptr) {
    if (!out || !ix || !offsets) { set_error("NULL argument"); return FMB_EINVAL; }
    *out = nullptr;
    const uint64_t mult = complement ? 2 : 1;
    if (nq * mult >= 0xFFFFFFFFull) { set_error("too many queries in one batch"); return FMB_EUNSUPPORTED; }
    FMB_TRY(use_device(ix->device));
    if (offsets[nq] < offsets[0]) { set_error("offsets not monotone"); return FMB_EINVAL; }
    const uint64_t in_total = offsets[nq] - offsets[0];
    if (in_total && !symbols && !pk) { set_error("symbols is NULL"); return FMB_EINVAL; }
    const uint64_t total = in_total * mult, nq_out = nq * mult;
    auto q = new fmb_queries();
    q->device = ix->device;
    q->nq = nq_out;
    q->total_symbols = total;
    cudaStream_t st = active_stream(ix);
    DevBuf<uint8_t> stage_sym;
    DevBuf<uint64_t> stage_off;
    int rc = q->symbols.alloc(total + 32);
    if (!rc) rc = q->offsets.alloc(nq_out + 1);
    if (!rc && complement) rc = stage_sym.alloc(in_total);
    if (!rc && complement) rc = stage_off.alloc(nq + 1);
    if (rc) { delete q; return rc; }
    uint8_t* sym_dst = complement ? stage_sym.p : q->symbols.p;
    uint64_t* off_dst = complement ? stage_off.p : q->offsets.p;
    cudaError_t e = cudaSuccess;
    DevBuf<uint32_t> stage_words;
    DevBuf<uint64_t> stage_epos;
    DevBuf<uint8_t> stage_esym;
    if (in_total && pk) {
        // only the 2-bit words of this slice cross PCIe (a quarter of the bytes); the byte symbols the kernels read are unpacked here
        const uint64_t first = offsets[0], w0 = first / 16, w1 = (first + in_total + 15) / 16;
        const uint64_t* lo = std::lower_bound(pk->exc_pos, pk->exc_pos + pk->n_exc, first);
        const uint64_t* hi = std::lower_bound(lo, pk->exc_pos + pk->n_exc, first + in_total);
        const uint64_t ne = (uint64_t)(hi - lo);
        rc = stage_words.alloc(w1 - w0);
        if (!rc && ne) rc = stage_epos.alloc(ne);
        if (!rc && ne) rc = stage_esym.alloc(ne);
        if (rc) { delete q; return rc; }
        q->h2d_bytes += (w1 - w0) * sizeof(uint32_t) + ne * 9;
        e = cudaMemcpyAsync(stage_words.p, pk->words + w0, (w1 - w0) * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess && ne) e = cudaMemcpyAsync(stage_epos.p, lo, ne * sizeof(uint64_t), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess && ne) e = cudaMemcpyAsync(stage_esym.p, pk->exc_sym + (lo - pk->exc_pos), ne, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) {
            unpack_queries_kernel<<<grid_for((in_total + 15) / 16, 256), 256, 0, st>>>(stage_words.p, first - w0 * 16, in_total, sym_dst);
            e = cudaGetLastError();
            note_launches(1);
        }
        if (e == cudaSuccess && ne) {
            apply_exceptions_kernel<<<grid_for(ne, 256), 256, 0, st>>>(stage_epos.p, stage_esym.p, ne, first, sym_dst);
            e = cudaGetLastError();
            note_launches(1);
        }
    } else if (in_total) {
        q->h2d_bytes += in_total;
        e = cudaMemcpyAsync(sym_dst, symbols + offsets[0], in_total, cudaMemcpyHostToDevice, st);
    }
    // validate the offsets while the symbols are in flight
    uint32_t mx = 0, mn = 0xFFFFFFFFu;
    for (uint64_t i = 0; i < nq; ++i) {
        if (offsets[i + 1] < offsets[i] || offsets[i + 1] - offsets[i] > 0xFFFFu) {
            set_error("query %llu: offsets not monotone or query longer than 65535", (unsigned long long)i);
            cudaStreamSynchronize(st);
            delete q;
            return FMB_EINVAL;
        }
        uint32_t L = (uint32_t)(offsets[i + 1] - offsets[i]);
        mx = std::max(mx, L);
        mn = std::min(mn, L);
    }
    q->max_len = mx;
    q->min_len = nq ? mn : 0;
    if (e == cudaSuccess) e = cudaMemsetAsync(q->symbols.p + total, 0xFF, 32, st);
    if (nq && mx == mn) {
        // reads of one length (the usual batch): offsets[i] = i * L is generated on the device, 8 bytes per query stay off PCIe
        if (e == cudaSuccess) {
            iota_offsets_kernel<<<grid_for(nq + 1, 256), 256, 0, st>>>(off_dst, nq + 1, mx);
            e = cudaGetLastError();
            note_launches(1);
        }
    } else {
        q->h2d_bytes += (nq + 1) * 8;
        if (e == cudaSuccess) e = cudaMemcpyAsync(off_dst, offsets, (nq + 1) * 8, cudaMemcpyHostToDevice, st);
    }
    if (e == cudaSuccess && offsets[0] != 0 && !(nq && mx == mn)) {
        // a slice of a larger batch: make the offsets relative to the first symbol of the slice, on the device
        rebase_offsets_kernel<<<grid_for(nq + 1, 256), 256, 0, st>>>(off_dst, nq + 1, offsets[0]);
        e = cudaGetLastError();
        note_launches(1);
    }
    if (e == cudaSuccess && complement) {
        ComplementTable ct;
        for (uint32_t c = 0; c < 32; ++c) ct.map[c] = c < ix->sigma ? complement[c] : (uint8_t)c;
        if (nq) {
            revcomp_double_kernel<<<grid_for(nq * 32, 256), 256, 0, st>>>(stage_sym.p, stage_off.p, nq, ct, q->symbols.p, q->offsets.p);
            e = cudaGetLastError();
            note_launches(1);
        } else {
            e = cudaMemsetAsync(q->offsets.p, 0, 8, st);
        }
    }
    if (e == cudaSuccess && ix->dna) {
        // 2-bit packed copy for the two-symbol / jump kernels
        const uint64_t words = (total + 15) / 16;
        rc = q->packed.alloc(words + 2);
        if (!rc) rc = q->flags.alloc(nq_out + 1);
        if (rc) { cudaStreamSynchronize(st); delete q; return rc; }
        e = cudaMemsetAsync(q->flags.p, 0, nq_out + 1, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(q->packed.p + words, 0, 2 * sizeof(uint32_t), st);
        if (e == cudaSuccess && words) {
            pack_queries_kernel<<<grid_for(words, 256), 256, 0, st>>>(q->symbols.p, total, q->offsets.p, nq_out, ix->sigma, q->packed.p, words, q->flags.p);
            e = cudaGetLastError();
            note_launches(1);
        }
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { set_error("query upload: %s", cudaGetErrorString(e)); delete q; return FMB_ECUDA; }
    *out = q;
    return FMB_OK;
}
int fmb_queries_upload(fmb_queries** out, const fmb_index* ix, const uint8_t* symbols, const uint64_t* offsets, uint64_t nq) {
    return upload_queries(out, ix, symbols, offsets, nq, nullptr);
}
int fmb_queries_upload_revcomp(fmb_queries** out, const fmb_index* ix, const uint8_t* symbols, const uint64_t* offsets, uint64_t nq, const uint8_t* complement) {
    if (!complement) { set_error("NULL complement table"); return FMB_EINVAL; }
    return upload_queries(out, ix, symbols, offsets, nq, complement);
}
int fmb_queries_upload_packed(fmb_queries** out, const fmb_index* ix, const uint32_t* packed, const uint64_t* offsets, uint64_t nq,
                              const uint64_t* exc_pos, const uint8_t* exc_sym, uint64_t n_exc) {
    if (!ix || !offsets) { set_error("NULL argument"); return FMB_EINVAL; }
    if (!ix->dna) { set_error("2-bit packed queries need an alphabet of at most 5 symbols (index has %u)", ix->sigma); return FMB_EUNSUPPORTED; }
    if ((offsets[nq] > offsets[0] && !packed) || (n_exc && (!exc_pos || !exc_sym))) { set_error("NULL argument"); return FMB_EINVAL; }
    PackedInput pk;
    pk.words = packed; pk.exc_pos = exc_pos; pk.exc_sym = exc_sym; pk.n_exc = n_exc;
    return upload_queries(out, ix, nullptr, offsets, nq, nullptr, &pk);
}
// host-side 2-bit packing (the input form of fmb_queries_upload_packed); plain C loop, the caller may split the range over threads
uint64_t fmb_pack_symbols(const uint8_t* symbols, uint64_t first, uint64_t count, uint32_t sigma, uint32_t* words,
                          uint64_t* exc_pos, uint8_t* exc_sym, uint64_t exc_capacity) {
    uint64_t n_exc = 0;
    const uint64_t end = first + count;
    uint64_t i = first;
    auto put = [&](uint64_t at) {
        const uint32_t s = symbols[at];
        if (s == 0 || s >= sigma) {
            if (n_exc < exc_capacity) { exc_pos[n_exc] = at; exc_sym[n_exc] = (uint8_t)s; }
            ++n_exc;
        }
        return (s - 1u) & 3u;
    };
    // leading partial word (first need not be a multiple of 16: the fields of other ranges in that word are left alone)
    while (i < end && (i & 15)) {
        const uint32_t sh = 2 * (uint32_t)(i & 15);
        words[i >> 4] = (words[i >> 4] & ~(3u << sh)) | (put(i) << sh);
        ++i;
    }
    for (; i + 16 <= end; i += 16) {
        uint32_t w = 0;
        for (uint32_t k = 0; k < 16; ++k) w |= put(i + k) << (2 * k);
        words[i >> 4] = w;
    }
    if (i < end) {
        uint32_t w = words[i >> 4];
        for (; i < end; ++i) {
            const uint32_t sh = 2 * (uint32_t)(i & 15);
            w = (w & ~(3u << sh)) | (put(i) << sh);
            words[i >> 4] = w;
        }
    }
    return n_exc;
}
void fmb_queries_destroy(fmb_queries* q) {
    if (!q) return;
    cudaSetDevice(q->device);
    delete q;
}
uint64_t fmb_queries_count(const fmb_queries* q) { return q ? q->nq : 0; }

// ---- exact search (K2) ---------------------------------------------------------------------------------------------
// The kernel writes one hit record per query (dense: len == 0 where the pattern does not occur), the interval lengths as the
// input of locate's scan, and counts hits / rows / line requests itself: ONE read-back of the counters ends the call.  The records
// are compacted (ascending qidx) only when a caller fetches them (fmb_results_fetch_hits).
int fmb_search_exact(const fmb_index* ix, const fmb_queries* q, fmb_results** out) {
    if (!ix || !q || !out) { set_error("NULL argument"); return FMB_EINVAL; }
    *out = nullptr;
    if (q->device != ix->device) { set_error("queries live on device %d, index on %d", q->device, ix->device); return FMB_EINVAL; }
    FMB_TRY(use_device(ix->device));
    cudaStream_t st = active_stream(ix);
    auto res = new fmb_results();
    res->device = ix->device;
    res->kind = 0;
    auto fail = [&](int rc) { delete res; return rc; };
    const uint64_t nq = q->nq;
    DevBuf<unsigned long long> ctr;
    int rc;
    if ((rc = res->hits.alloc(nq)) || (rc = res->lens.alloc(nq + 1)) || (rc = ctr.alloc(8))) return fail(rc);
    const bool two = ix->dna && ix->occ2.p && q->packed.p && ix->exact_mode != FMB_EXACT_ONE_SYMBOL;
    Occ2View o2 = ix->view_occ2();
    if (ix->exact_mode == FMB_EXACT_NO_TEXT) o2.isa = nullptr;
    // (seq, pos) of the hits the text check finds, for locate: only written when locate can use them
    const bool want_at = two && o2.isa && ix->text_rate && nq;
    if (want_at && (rc = res->at.alloc(nq))) return fail(rc);
    if (ix->exact_mode == FMB_EXACT_TWO_SYMBOL && !ix->occ2.p) { set_error("index has no two-symbol table"); return fail(FMB_EUNSUPPORTED); }
    cudaMemsetAsync(ctr.p, 0, 8 * sizeof(unsigned long long), st);
    cudaMemsetAsync(res->lens.p + nq, 0, sizeof(uint32_t), st);
    EventTimer tm(st);
    if (nq) {
        const uint32_t base = (uint32_t)q->qidx_base;
        if (two) exact_search2_kernel<<<grid_for(nq * 4, 256), 256, 0, st>>>(ix->view_dna(), o2, q->symbols.p, q->packed.p, q->flags.p, q->offsets.p, (uint32_t)nq, base, res->hits.p, res->lens.p,
                                                                             want_at ? res->at.p : nullptr, ctr.p);
        // (the one-symbol mode counts the algorithmic work: a four-symbol jump that fails counts four steps where the walk stops at the
        //  first mismatch, so that mode takes no jumps on the generic layout either)
        else FMB_DISPATCH(ix, v, exact_search_kernel<<<grid_for(nq, 256), 256, 0, st>>>(v, q->symbols.p, q->offsets.p, (uint32_t)nq, base, res->hits.p, res->lens.p, ctr.p,
                                                                                              ix->dna || ix->exact_mode == FMB_EXACT_ONE_SYMBOL ? nullptr : ix->jump4[0].p));
        note_launches(1);
    }
    unsigned long long h_ctr[8] = {0};
    cudaMemcpyAsync(h_ctr, ctr.p, sizeof h_ctr, cudaMemcpyDeviceToHost, st);
    const double ms = tm.stop();            // synchronises the stream: kernel and read-back are done
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("exact search: %s", cudaGetErrorString(e)); return fail(FMB_ECUDA); }
    res->stats.kernel_ms = ms;
    res->stats.main_kernel_ms = nq ? ms : 0.0;
    res->stats.extensions = h_ctr[0];
    res->stats.occ_lookups = h_ctr[1];
    res->stats.line_requests = h_ctr[2];
    res->count = h_ctr[4];
    res->total_rows = h_ctr[5];
    res->slots = nq;
    res->dense = true;
    *out = res;
    return FMB_OK;
}

// ---- locate (K4) ------------------------------------------------------------------------------------------------
int fmb_locate(const fmb_index* ix, const fmb_results* hits, fmb_results** out) {
    if (!ix || !hits || !out) { set_error("NULL argument"); return FMB_EINVAL; }
    *out = nullptr;
    if (hits->kind != 0) { set_error("fmb_locate needs a hit result set"); return FMB_EINVAL; }
    if (hits->device != ix->device) { set_error("results live on another device"); return FMB_EINVAL; }
    if (hits->count && ix->n_samples == 0) { set_error("index has no sampled suffix array: locate is impossible"); return FMB_EINVAL; }
    FMB_TRY(use_device(ix->device));
    cudaStream_t st = active_stream(ix);
    auto res = new fmb_results();
    res->device = ix->device;
    res->kind = 1;
    auto fail = [&](int rc) { delete res; return rc; };
    const uint64_t nh = hits->dense ? hits->slots : hits->count;       // records (dense: one per query, len 0 allowed)
    DevBuf<uint32_t> starts;
    DevBuf<unsigned long long> ctr, d_sum;
    DevBuf<uint8_t> tmp;
    int rc;
    if ((rc = starts.alloc(nh + 1)) || (rc = ctr.alloc(4))) return fail(rc);
    cudaMemsetAsync(ctr.p, 0, 4 * sizeof(unsigned long long), st);
    EventTimer tm(st);
    const uint32_t* lens = hits->lens.p;
    if (!lens) {
        hit_lengths_kernel<<<grid_for(nh + 1, 256), 256, 0, st>>>(hits->hits.p, nh, starts.p);
        note_launches(1);
        lens = starts.p;
    }
    // rows are numbered with 32 bits on the device: refuse (loudly) a result set whose intervals sum to 2^32 rows or more.  The search
    // kernels count the rows of their hits themselves; only result sets of unknown total need a reduction (and a round trip) here.
    unsigned long long h_sum = hits->total_rows;
    if (h_sum == UINT64_MAX) {
        if ((rc = d_sum.alloc(1))) return fail(rc);
        size_t tmp_bytes = 0;
        cub::TransformInputIterator<unsigned long long, ToU64, const uint32_t*> it(lens, ToU64{});
        cub::DeviceReduce::Sum(nullptr, tmp_bytes, it, d_sum.p, (int64_t)(nh + 1), st);
        DevBuf<uint8_t> rtmp;
        if ((rc = rtmp.alloc(tmp_bytes))) return fail(rc);
        cub::DeviceReduce::Sum(rtmp.p, tmp_bytes, it, d_sum.p, (int64_t)(nh + 1), st);
        if (cudaMemcpyAsync(&h_sum, d_sum.p, sizeof h_sum, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) {
            set_error("locate: row count failed");
            return fail(FMB_ECUDA);
        }
    }
    if (h_sum >= 0xFFFFFFFFull) {
        set_error("locate: the hits cover %llu rows; this build locates fewer than 2^32 rows per call -- split the batch", h_sum);
        return fail(FMB_EOVERFLOW);
    }
    const uint32_t total = (uint32_t)h_sum;
    // every record exactly one row: record h is row h, no scan and no binary search
    const bool single = total == nh && hits->count == nh;
    if (!single) {
        size_t tmp_bytes = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, lens, starts.p, (int64_t)(nh + 1), st);
        if ((rc = tmp.alloc(tmp_bytes))) return fail(rc);              // lives until the stream is synchronised below
        cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, lens, starts.p, (int64_t)(nh + 1), st);
        note_launches(1);
    }
    if ((rc = res->locs.alloc(total))) return fail(rc);
    cudaEvent_t ev_m0 = nullptr, ev_m1 = nullptr;
    cudaEventCreate(&ev_m0);
    cudaEventCreate(&ev_m1);
    if (total) {
        cudaEventRecord(ev_m0, st);
        if ((ix->sa.p || ix->locrow.p) && ix->locate_mode != FMB_LOCATE_WALK) {
            const uint2* at = hits->dense && ix->text_rate ? hits->at.p : nullptr;
            locate_shortcut_kernel<<<grid_for(total, 256), 256, 0, st>>>(ix->view_rowpos(), hits->hits.p, starts.p, (uint32_t)nh, total, single ? 1u : 0u, at,
                                                                         res->locs.p, ctr.p);
        } else if (ix->dna && ix->locblocks.p) {
            auto v = ix->view_dna();
            // persistent grid: every SM full of lane pairs (8 blocks x 256 threads), rows handed out with a grid stride
            const int sms = ix->sm_count;
            unsigned grid = (unsigned)std::min<uint64_t>(grid_for((uint64_t)total * 2, 256), (uint64_t)sms * 8);
            locate_pair_kernel<<<grid, 256, 0, st>>>(v, hits->hits.p, starts.p, (uint32_t)nh, total, single ? 1u : 0u, res->locs.p, ctr.p);
        }
        else FMB_DISPATCH(ix, v, locate_kernel<<<grid_for(total, 256), 256, 0, st>>>(v, hits->hits.p, starts.p, (uint32_t)nh, total, single ? 1u : 0u, res->locs.p, ctr.p));
        cudaEventRecord(ev_m1, st);
        note_launches(1);
    }
    unsigned long long h_ctr[4] = {0};
    cudaMemcpyAsync(h_ctr, ctr.p, sizeof h_ctr, cudaMemcpyDeviceToHost, st);
    res->stats.kernel_ms = tm.stop();       // synchronises the stream
    if (total) {
        float ms = 0;
        cudaEventElapsedTime(&ms, ev_m0, ev_m1);
        res->stats.main_kernel_ms = ms;
    }
    cudaEventDestroy(ev_m0);
    cudaEventDestroy(ev_m1);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("locate: %s", cudaGetErrorString(e)); return fail(FMB_ECUDA); }
    res->stats.lf_steps = h_ctr[2];
    res->stats.occ_lookups = h_ctr[1];
    res->count = total;
    res->slots = total;
    *out = res;
    return FMB_OK;
}

int fmb_locate_rows(const fmb_index* ix, const uint64_t* rows, uint64_t count, uint32_t* seq, uint32_t* pos, uint64_t* steps) {
    if (!ix || (count && (!rows || !seq || !pos || !steps))) { set_error("NULL argument"); return FMB_EINVAL; }
    FMB_TRY(use_device(ix->device));
    if (count == 0) return FMB_OK;
    if (ix->n_samples == 0) { set_error("index has no sampled suffix array"); return FMB_EINVAL; }
    for (uint64_t i = 0; i < count; ++i)
        if (rows[i] >= ix->n) { set_error("rows[%llu] = %llu out of range", (unsigned long long)i, (unsigned long long)rows[i]); return FMB_EINVAL; }
    cudaStream_t st = active_stream(ix);
    DevBuf<uint64_t> d_rows, d_steps;
    DevBuf<uint32_t> d_seq, d_pos;
    FMB_TRY(upload(d_rows, rows, count, st));
    FMB_TRY(d_steps.alloc(count));
    FMB_TRY(d_seq.alloc(count));
    FMB_TRY(d_pos.alloc(count));
    FMB_DISPATCH(ix, v, locate_rows_kernel<<<grid_for(count, 256), 256, 0, st>>>(v, d_rows.p, count, d_seq.p, d_pos.p, d_steps.p));
    FMB_CUDA(cudaGetLastError());
    note_launches(1);
    FMB_CUDA(cudaMemcpyAsync(seq, d_seq.p, count * 4, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaMemcpyAsync(pos, d_pos.p, count * 4, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaMemcpyAsync(steps, d_steps.p, count * 8, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    return FMB_OK;
}

int fmb_sample_value(const fmb_index* ix, const uint64_t* rows, uint64_t count, uint8_t* has, uint32_t* seq, uint32_t* pos) {
    if (!ix || (count && (!rows || !has || !seq || !pos))) { set_error("NULL argument"); return FMB_EINVAL; }
    FMB_TRY(use_device(ix->device));
    if (count == 0) return FMB_OK;
    for (uint64_t i = 0; i < count; ++i)
        if (rows[i] >= ix->n) { set_error("rows[%llu] = %llu out of range", (unsigned long long)i, (unsigned long long)rows[i]); return FMB_EINVAL; }
    cudaStream_t st = active_stream(ix);
    DevBuf<uint64_t> d_rows;
    DevBuf<uint32_t> d_seq, d_pos;
    DevBuf<uint8_t> d_has;
    FMB_TRY(upload(d_rows, rows, count, st));
    FMB_TRY(d_has.alloc(count));
    FMB_TRY(d_seq.alloc(count));
    FMB_TRY(d_pos.alloc(count));
    FMB_DISPATCH(ix, v, sample_value_kernel<<<grid_for(count, 256), 256, 0, st>>>(v, d_rows.p, count, d_has.p, d_seq.p, d_pos.p));
    FMB_CUDA(cudaGetLastError());
    note_launches(1);
    FMB_CUDA(cudaMemcpyAsync(has, d_has.p, count, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaMemcpyAsync(seq, d_seq.p, count * 4, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaMemcpyAsync(pos, d_pos.p, count * 4, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    return FMB_OK;
}

// ---- results ----------------------------------------------------------------------------------------------------
uint64_t fmb_results_count(const fmb_results* r) { return r ? r->count : 0; }
int fmb_results_kind(const fmb_results* r) { return r ? r->kind : -1; }

int fmb_results_fetch_hits(const fmb_results* r, fmb_hit* out, uint64_t capacity) {
    if (!r || (!out && r->count)) { set_error("NULL argument"); return FMB_EINVAL; }
    if (r->kind != 0) { set_error("result set holds no hits (kind %d)", r->kind); return FMB_EINVAL; }
    if (capacity < r->count) { set_error("capacity %llu < %llu hits", (unsigned long long)capacity, (unsigned long long)r->count); return FMB_EOVERFLOW; }
    FMB_TRY(use_device(r->device));
    const uint64_t slots = r->dense ? r->slots : r->count;
    std::vector<HitRec> h(slots);
    if (slots) FMB_CUDA(cudaMemcpy(h.data(), r->hits.p, slots * sizeof(HitRec), cudaMemcpyDeviceToHost));
    uint64_t k = 0;
    for (uint64_t i = 0; i < slots; ++i) {
        if (r->dense && h[i].len == 0) continue;                   // dense results: queries without hit have an empty record
        if (k < r->count) out[k] = fmb_hit{h[i].qidx, h[i].lb, h[i].lb_rev, h[i].len, h[i].steps, h[i].e};
        ++k;
    }
    if (k != r->count) { set_error("result set is inconsistent: %llu records, %llu counted", (unsigned long long)k, (unsigned long long)r->count); return FMB_ECUDA; }
    return FMB_OK;
}
int fmb_results_fetch_locs32(const fmb_results* r, fmb_loc32* out, uint64_t capacity) {
    if (!r || (!out && r->count)) { set_error("NULL argument"); return FMB_EINVAL; }
    if (r->kind != 1) { set_error("result set holds no located rows (kind %d)", r->kind); return FMB_EINVAL; }
    if (capacity < r->count) { set_error("capacity %llu < %llu rows", (unsigned long long)capacity, (unsigned long long)r->count); return FMB_EOVERFLOW; }
    FMB_TRY(use_device(r->device));
    if (r->count) FMB_CUDA(cudaMemcpy(out, r->locs.p, r->count * sizeof(LocRec), cudaMemcpyDeviceToHost));
    return FMB_OK;
}
int fmb_results_fetch_locs(const fmb_results* r, fmb_loc* out, uint64_t capacity) {
    if (!r || (!out && r->count)) { set_error("NULL argument"); return FMB_EINVAL; }
    if (r->kind != 1) { set_error("result set holds no located rows (kind %d)", r->kind); return FMB_EINVAL; }
    if (capacity < r->count) { set_error("capacity too small"); return FMB_EOVERFLOW; }
    std::vector<fmb_loc32> h(r->count);
    FMB_TRY(fmb_results_fetch_locs32(r, h.data(), r->count));
    for (uint64_t i = 0; i < r->count; ++i) out[i] = fmb_loc{h[i].qidx, h[i].seq, h[i].pos, h[i].e};
    return FMB_OK;
}
int fmb_results_get_stats(const fmb_results* r, fmb_stats* out) {
    if (!r || !out) { set_error("NULL argument"); return FMB_EINVAL; }
    *out = r->stats;
    return FMB_OK;
}
void fmb_results_destroy(fmb_results* r) {
    if (!r) return;
    cudaSetDevice(r->device);
    delete r;
}

// ---- helpers ------------------------------------------------------------------------------------------------------
int fmb_synth_text_device(int device, uint32_t sigma, uint64_t n, uint64_t seed, uint8_t** d_text) {
    if (!d_text || sigma < 2 || n == 0) { set_error("bad argument"); return FMB_EINVAL; }
    FMB_TRY(use_device(device));
    uint8_t* p = nullptr;
    FMB_TRY(raw_alloc(&p, n));
    synth_text_kernel<<<grid_for(n, 256), 256>>>(p, n, sigma, seed);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaDeviceSynchronize());
    *d_text = p;
    return FMB_OK;
}
int fmb_synth_reads_device(int device, const uint8_t* d_text, uint64_t n, uint64_t nq, uint32_t length, uint64_t seed, uint8_t** d_reads) {
    if (!d_text || !d_reads || length == 0 || n <= (uint64_t)length + 1) { set_error("bad argument"); return FMB_EINVAL; }
    FMB_TRY(use_device(device));
    uint8_t* p = nullptr;
    FMB_TRY(raw_alloc(&p, nq * length + 32));
    synth_reads_kernel<<<grid_for(nq * length, 256), 256>>>(d_text, n, nq, length, seed, p);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaDeviceSynchronize());
    *d_reads = p;
    return FMB_OK;
}
int fmb_synth_repeat_text_device(int device, uint32_t sigma, uint64_t n, uint64_t seed, uint32_t unit_len, uint32_t copies,
                                 uint32_t sub_per_mille, uint8_t** d_text) {
    if (!d_text || sigma < 3 || copies == 0 || unit_len == 0 || (n - 1) / copies <= (uint64_t)unit_len + 1) { set_error("bad argument"); return FMB_EINVAL; }
    FMB_TRY(fmb_synth_text_device(device, sigma, n, seed, d_text));
    splice_repeats_kernel<<<grid_for((uint64_t)copies * unit_len, 256), 256>>>(*d_text, n, sigma, seed, unit_len, copies, sub_per_mille);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaDeviceSynchronize());
    return FMB_OK;
}
int fmb_synth_unit_reads_device(int device, uint32_t sigma, uint64_t nq, uint32_t length, uint64_t seed, uint32_t unit_len, uint8_t** d_reads) {
    if (!d_reads || length == 0 || unit_len <= length || sigma < 3) { set_error("bad argument"); return FMB_EINVAL; }
    FMB_TRY(use_device(device));
    uint8_t* p = nullptr;
    FMB_TRY(raw_alloc(&p, nq * length + 32));
    unit_reads_kernel<<<grid_for(nq * length, 256), 256>>>(nq, length, seed, unit_len, sigma, p);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaDeviceSynchronize());
    *d_reads = p;
    return FMB_OK;
}
int fmb_synth_reads_err_device(int device, const uint8_t* d_text, uint64_t n, uint64_t nq, uint32_t length, uint64_t seed,
                               uint32_t sigma, uint32_t max_errors, int edit, uint8_t** d_reads) {
    if (!d_text || !d_reads || length < 3 || length > 512 || sigma < 3 || n <= (uint64_t)length + 1) { set_error("bad argument"); return FMB_EINVAL; }
    FMB_TRY(use_device(device));
    uint8_t* p = nullptr;
    FMB_TRY(raw_alloc(&p, nq * length + 32));
    synth_reads_err_kernel<<<grid_for(nq, 128), 128>>>(d_text, n, nq, length, seed, max_errors, edit ? 1u : 0u, sigma, p);
    FMB_CUDA(cudaGetLastError());
    FMB_CUDA(cudaDeviceSynchronize());
    *d_reads = p;
    return FMB_OK;
}
// Empirical random-access ceiling of THIS device over one of the index's own tables (SURVEY.md §8d): independent random gathers,
// one request per granule, timed with CUDA events on the index's stream.
int fmb_measure_gather(const fmb_index* ix, int table, uint64_t requests, double* requests_per_s, uint64_t* table_bytes, uint32_t* request_bytes) {
    if (!ix || !requests_per_s) { set_error("NULL argument"); return FMB_EINVAL; }
    FMB_TRY(use_device(ix->device));
    cudaStream_t st = active_stream(ix);
    const char* tab = nullptr;
    uint64_t bytes = 0;
    uint32_t per = 0, lanes = 0;
    switch (table) {
        case FMB_GATHER_PAIR_LINE: tab = (const char*)ix->occ2.p; bytes = (ix->n / 128 + 1) * 128; per = 32; lanes = 4; break;
        case FMB_GATHER_OCC_BLOCK:
            if (ix->dna) { tab = (const char*)ix->occ_dna[0].p; bytes = (ix->n / 64 + 1) * 32; per = 32; lanes = 1; }
            else { tab = (const char*)ix->occ_gen[0].p; bytes = (ix->n / 64 + 1) * (uint64_t)ix->gen_stride; per = 32; lanes = ix->gen_stride / 32; }
            break;
        case FMB_GATHER_JUMP_ENTRY:
            if (ix->jump[0].p) { tab = (const char*)ix->jump[0].p; per = ix->jump_shift[0] ? 16 : 8; bytes = ix->n * per; lanes = 1; }
            else if (ix->jump4[0].p) { tab = (const char*)ix->jump4[0].p; per = 8; bytes = ix->n * 8; lanes = 1; }
            break;
        default: set_error("unknown table %d", table); return FMB_EINVAL;
    }
    if (!tab || !(lanes == 1 || lanes == 2 || lanes == 4)) { set_error("the index has no such table"); return FMB_EUNSUPPORTED; }
    int sms = 0;
    FMB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ix->device));
    const uint64_t groups = (uint64_t)sms * 8 * 256 / lanes;
    const uint32_t iters = (uint32_t)std::max<uint64_t>(4, (requests + groups - 1) / groups / 4 * 4);
    const uint64_t ngran = bytes / ((uint64_t)per * lanes);
    DevBuf<uint32_t> sink;
    FMB_TRY(sink.alloc(1));
    auto launch = [&]() {
        const unsigned grid = (unsigned)(sms * 8);
        if (per == 8) gather_probe_kernel<8, 1><<<grid, 256, 0, st>>>(tab, ngran, iters, sink.p);
        else if (per == 16) gather_probe_kernel<16, 1><<<grid, 256, 0, st>>>(tab, ngran, iters, sink.p);
        else if (lanes == 1) gather_probe_kernel<32, 1><<<grid, 256, 0, st>>>(tab, ngran, iters, sink.p);
        else if (lanes == 2) gather_probe_kernel<32, 2><<<grid, 256, 0, st>>>(tab, ngran, iters, sink.p);
        else gather_probe_kernel<32, 4><<<grid, 256, 0, st>>>(tab, ngran, iters, sink.p);
        note_launches(1);
    };
    launch();                                   // warm-up (TLB, clocks)
    FMB_CUDA(cudaStreamSynchronize(st));
    double best = 1e30;
    for (int rep = 0; rep < 3; ++rep) {
        EventTimer tm(st);
        launch();
        best = std::min(best, tm.stop());
    }
    FMB_CUDA(cudaGetLastError());
    *requests_per_s = (double)groups * iters / (best * 1e-3);
    if (table_bytes) *table_bytes = bytes;
    if (request_bytes) *request_bytes = per * lanes;
    return FMB_OK;
}

int fmb_set_image_budget(uint64_t bytes) {
    g_image_budget.store(bytes);
    return FMB_OK;
}
int fmb_index_set_stream(fmb_index* ix, void* stream) {
    if (!ix) { set_error("NULL index"); return FMB_EINVAL; }
    ix->stream = stream ? (cudaStream_t)stream : ix->own_stream;
    return FMB_OK;
}
int fmb_index_set_exact_mode(fmb_index* ix, int mode) {
    if (!ix || mode < 0 || mode > 3) { set_error("bad argument"); return FMB_EINVAL; }
    if ((mode == FMB_EXACT_TWO_SYMBOL || mode == FMB_EXACT_NO_TEXT) && !ix->occ2.p) { set_error("index has no two-symbol table"); return FMB_EUNSUPPORTED; }
    ix->exact_mode = mode;
    return FMB_OK;
}
int fmb_index_set_locate_mode(fmb_index* ix, int mode) {
    if (!ix || mode < 0 || mode > 1) { set_error("bad argument"); return FMB_EINVAL; }
    ix->locate_mode = mode;
    return FMB_OK;
}
uint64_t fmb_kernel_launch_count(void) { return fmb::g_launches.load(); }
int fmb_device_free(int device, void* p) {
    FMB_TRY(use_device(device));
    FMB_CUDA(cudaFree(p));
    return FMB_OK;
}
int fmb_copy_to_host(int device, void* dst_host, const void* src_device, uint64_t bytes) {
    FMB_TRY(use_device(device));
    FMB_CUDA(cudaMemcpy(dst_host, src_device, bytes, cudaMemcpyDeviceToHost));
    return FMB_OK;
}
void* fmb_host_alloc_pinned(uint64_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); set_error("cudaMallocHost(%llu) failed", (unsigned long long)bytes); return nullptr; }
    return p;
}
void fmb_host_free_pinned(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
