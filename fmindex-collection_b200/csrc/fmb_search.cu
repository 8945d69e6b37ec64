// fmb_search.cu -- host side of the k-error searches (K3) and the one-call search+locate path.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cub/cub.cuh>

#include "fmb_host.hpp"
#include "fmb_scheme.cuh"
#include "fmb_text.cuh"

using namespace fmb;

namespace {

int set_device(int device) {
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cudaSetDevice(%d): %s -- libfmb200 has no CPU fallback", device, cudaGetErrorString(e));
        return FMB_ENODEVICE;
    }
    return FMB_OK;
}

constexpr uint32_t kStackCapDefault = 160;   // items per warp (5 KB; 40 KB per block, 4 blocks per SM)
constexpr uint32_t kWarpsPerBlock = 8;
constexpr int kMaxDevices = 64;

struct EventPair {          // the two timing events of a search call, destroyed on every exit path
    cudaEvent_t a = nullptr, b = nullptr;
    EventPair() { cudaEventCreate(&a); cudaEventCreate(&b); }
    ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    EventPair(const EventPair&) = delete;
    EventPair& operator=(const EventPair&) = delete;
};

JumpView make_jump_view(const fmb_index* ix, const fmb_queries* q) {
    JumpView jv{};
    static const bool no_jump = getenv("FMB_NO_SCHEME_JUMP") != nullptr;
    if (!ix->dna && !no_jump) {
        jv.jump4[0] = ix->jump4[0].p;         // byte-symbol LF^4 tables of the generic layout
        jv.jump4[1] = ix->jump4[1].p;
        jv.bikmer = ix->bikmer.p;             // ... and its bidirectional k-mer table (index = base-(sigma - first_symb) number)
        jv.bikmer_k = ix->bikmer.p ? ix->bikmer_k : 0;
        jv.bikmer_base = ix->sigma - ix->first_symb;
    }
    if (ix->dna && q->packed.p && !no_jump) {
        jv.jump[0] = ix->jump[0].p;
        jv.jump[1] = ix->jump[1].p;
        jv.jshift[0] = ix->jump_shift[0];
        jv.jshift[1] = ix->jump_shift[1];
        jv.jump4[0] = ix->jump4[0].p;
        jv.jump4[1] = ix->jump4[1].p;
        jv.qpk = q->packed.p;
        jv.qflags = q->flags.p;
        jv.bikmer = ix->bikmer.p;
        jv.bikmer_k = ix->bikmer.p ? ix->bikmer_k : 0;
    }
    return jv;
}

// edit-distance searches decide single-row intervals on the text (scheme_text_kernel) when the index holds the tables that serve as
// text windows in both directions: LF^16 entries (sigma <= 5, 2-bit packed queries) or byte-symbol LF^4 entries (generic layout)
bool text_mode_available(const fmb_index* ix, const fmb_queries* q, bool left_only) {
    static const bool off = getenv("FMB_NO_TEXT") != nullptr;
    if (off) return false;
    const JumpView jv = make_jump_view(ix, q);
    return ix->dna ? (jv.jump[0] && (left_only || jv.jump[1]) && jv.qpk) : (jv.jump4[0] && (left_only || jv.jump4[1]));
}

template <class OCC, bool EDIT, bool PSEUDO>
int launch_text_t(const fmb_index* ix, const IndexView<OCC>& view, const SchemeParams& sp, const fmb_queries* q, const Item* items, uint64_t n_items,
                  const SchemeOut& out, cudaStream_t st) {
    auto kern = scheme_text_kernel<OCC, EDIT, PSEUDO>;
    static std::mutex cfg_mu;
    static int cfg_blocks_per_sm[kMaxDevices] = {};
    int blocks_per_sm;
    {
        std::lock_guard<std::mutex> lk(cfg_mu);
        const int dev = ix->device;
        if (dev < 0 || dev >= kMaxDevices) { set_error("device %d outside [0,%d)", dev, kMaxDevices); return FMB_EINVAL; }
        if (!cfg_blocks_per_sm[dev]) {
            int bps = 0;
            FMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, 256, 0));
            cfg_blocks_per_sm[dev] = bps < 1 ? 1 : bps;
        }
        blocks_per_sm = cfg_blocks_per_sm[dev];
    }
    const uint64_t want_blocks = (n_items + 255) / 256;
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)ix->sm_count * blocks_per_sm, want_blocks));
    kern<<<grid, 256, 0, st>>>(view, sp, q->symbols.p, q->offsets.p, make_jump_view(ix, q), items, n_items, out);
    FMB_CUDA(cudaGetLastError());
    note_launches(1);
    return FMB_OK;
}
int launch_text(const fmb_index* ix, const SchemeParams& sp, const fmb_queries* q, const Item* items, uint64_t n_items, const SchemeOut& out, bool pseudo,
                cudaStream_t st) {
    if (!sp.edit) return ix->dna ? launch_text_t<OccDna, false, false>(ix, ix->view_dna(), sp, q, items, n_items, out, st)
                                 : launch_text_t<OccGen, false, false>(ix, ix->view_gen(), sp, q, items, n_items, out, st);
    if (ix->dna) return pseudo ? launch_text_t<OccDna, true, true>(ix, ix->view_dna(), sp, q, items, n_items, out, st)
                               : launch_text_t<OccDna, true, false>(ix, ix->view_dna(), sp, q, items, n_items, out, st);
    return pseudo ? launch_text_t<OccGen, true, true>(ix, ix->view_gen(), sp, q, items, n_items, out, st)
                  : launch_text_t<OccGen, true, false>(ix, ix->view_gen(), sp, q, items, n_items, out, st);
}

// FMB_SCHEME_CAP: items per warp stack of the frontier kernel (read once per process).  A warp takes roots 32 at a time, so a stack of
// fewer than 32 items could never take one, and a block whose stacks exceed the device's shared memory cannot launch: both are
// refused before any launch.
int scheme_stack_cap(int dev, size_t item_bytes, uint32_t* cap) {
    static const char* env = getenv("FMB_SCHEME_CAP");
    unsigned long long v = kStackCapDefault;
    if (env) {
        char* end = nullptr;
        v = strtoull(env, &end, 10);
        if (end == env || *end != '\0') { set_error("FMB_SCHEME_CAP=%s is not a number", env); return FMB_EINVAL; }
    }
    int smem_max = 0;
    FMB_CUDA(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    const unsigned long long v_max = (unsigned long long)smem_max / (kWarpsPerBlock * item_bytes);
    if (v < 32 || v > v_max) {
        set_error("FMB_SCHEME_CAP=%llu: the frontier kernel's warp stacks hold 32..%llu items on device %d", v, v_max, dev);
        return FMB_EINVAL;
    }
    *cap = (uint32_t)v;
    return FMB_OK;
}

template <class OCC, bool EDIT, bool ORDERED, bool PSEUDO>
int launch_frontier_t(const fmb_index* ix, const IndexView<OCC>& view, const SchemeParams& sp, const fmb_queries* q, uint64_t n_roots, const Item* in_items,
                      uint64_t n_in, const SchemeOut& out, cudaStream_t st) {
    constexpr size_t kItemBytes = sizeof(Item) + (ORDERED ? sizeof(unsigned long long) : 0);
    auto kern = scheme_search_kernel<OCC, EDIT, ORDERED, PSEUDO>;
    // launch geometry, computed once per kernel instantiation (several host threads drive one index in the pipelined path)
    // (cached per device: several replicas of an index may be driven from concurrent threads, fmb200/multi.hpp)
    static std::mutex cfg_mu;
    static int cfg_blocks_per_sm[kMaxDevices] = {}, cfg_sms[kMaxDevices] = {};
    static uint32_t cfg_cap[kMaxDevices] = {};
    int blocks_per_sm, sms;
    uint32_t stack_cap;
    size_t smem;
    {
        std::lock_guard<std::mutex> lk(cfg_mu);
        const int dev = ix->device;
        if (dev < 0 || dev >= kMaxDevices) { set_error("device %d outside [0,%d)", dev, kMaxDevices); return FMB_EINVAL; }
        if (!cfg_cap[dev]) FMB_TRY(scheme_stack_cap(dev, kItemBytes, &cfg_cap[dev]));
        stack_cap = cfg_cap[dev];
        smem = (size_t)stack_cap * kWarpsPerBlock * kItemBytes;
        FMB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));      // per device
        if (!cfg_blocks_per_sm[dev]) {
            int bps = 0;
            FMB_CUDA(cudaDeviceGetAttribute(&cfg_sms[dev], cudaDevAttrMultiProcessorCount, dev));
            FMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, 256, smem));
            cfg_blocks_per_sm[dev] = bps < 1 ? 1 : bps;
        }
        blocks_per_sm = cfg_blocks_per_sm[dev];
        sms = cfg_sms[dev];
    }
    uint64_t work = n_roots + n_in;
    uint64_t want_blocks = (work + 255) / 256;
    unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)sms * blocks_per_sm, want_blocks));
    const JumpView jv = make_jump_view(ix, q);
    kern<<<grid, 256, smem, st>>>(view, sp, q->symbols.p, q->offsets.p, jv, n_roots, in_items, n_in, out, stack_cap);
    FMB_CUDA(cudaGetLastError());
    note_launches(1);
    return FMB_OK;
}
template <class OCC>
int launch_frontier_v(const fmb_index* ix, const IndexView<OCC>& v, const SchemeParams& sp, const fmb_queries* q, bool ordered, bool pseudo,
                      uint64_t n_roots, const Item* in_items, uint64_t n_in, const SchemeOut& out, cudaStream_t st) {
    if (ordered) return sp.edit ? launch_frontier_t<OCC, true, true, false>(ix, v, sp, q, n_roots, in_items, n_in, out, st)
                                : launch_frontier_t<OCC, false, true, false>(ix, v, sp, q, n_roots, in_items, n_in, out, st);
    if (!sp.edit) return launch_frontier_t<OCC, false, false, false>(ix, v, sp, q, n_roots, in_items, n_in, out, st);
    return pseudo ? launch_frontier_t<OCC, true, false, true>(ix, v, sp, q, n_roots, in_items, n_in, out, st)
                  : launch_frontier_t<OCC, true, false, false>(ix, v, sp, q, n_roots, in_items, n_in, out, st);
}
// ordered: the hit-limited instantiation (discovery-order keys); pseudo: edit distance without the redundancy filter
int launch_frontier(const fmb_index* ix, const SchemeParams& sp, const fmb_queries* q, bool ordered, bool pseudo, uint64_t n_roots,
                    const Item* in_items, uint64_t n_in, const SchemeOut& out, cudaStream_t st) {
    if (ix->dna) return launch_frontier_v(ix, ix->view_dna(), sp, q, ordered, pseudo, n_roots, in_items, n_in, out, st);
    return launch_frontier_v(ix, ix->view_gen(), sp, q, ordered, pseudo, n_roots, in_items, n_in, out, st);
}

// ---- text list by class: the lanes of a warp of the text kernel take consecutive items; items of one (search, part, errors) class
//      run the same branches of the state machine (skippable stretch, 16-position evaluation, node visits), so the list is grouped
//      by class before the kernel reads it (one 8-bit radix pass over 4-byte keys + a gather; ~0.3 ms per 8 M items)
__global__ void text_class_keys_kernel(const Item* __restrict__ items, uint64_t count, uint32_t* __restrict__ keys, uint32_t* __restrict__ idx) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t meta = items[i].meta;
    // search (4 bits of it), part (4 bits), errors so far (2 bits): 10 bits
    keys[i] = (((meta >> 16) & 15u) << 6) | (((meta >> 8) & 15u) << 2) | (meta & 3u);
    idx[i] = (uint32_t)i;
}
__global__ void gather_items_kernel(const Item* __restrict__ items, const uint32_t* __restrict__ idx, uint64_t count, Item* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < count) out[i] = items[idx[i]];
}

// ---- hit limit: put the hits into the reference's discovery order and cut every query off after n rows ----------------------
__global__ void iota_kernel(uint32_t* out, uint64_t count) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < count) out[i] = (uint32_t)i;
}
__global__ void gather_qidx_kernel(const HitRec* __restrict__ hits, const uint32_t* __restrict__ perm, uint32_t* __restrict__ out, uint64_t count) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < count) out[i] = hits[perm[i]].qidx;
}
__global__ void gather_hits_kernel(const HitRec* __restrict__ hits, const uint32_t* __restrict__ perm, HitRec* __restrict__ out, uint64_t count) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < count) out[i] = hits[perm[i]];
}
// search_n_impl's delegate (SearchNg26.h:414-421): `ct` rows reported so far; a cursor that would exceed n is clipped to n - ct rows,
// and the query ends when ct == n.  hits are sorted by (qidx, discovery order); the thread at the first hit of a query walks
// that query's hits (flags are zero beforehand).
__global__ void limit_rows_kernel(HitRec* __restrict__ hits, uint32_t* __restrict__ keep, uint64_t count, unsigned long long n) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t q = hits[i].qidx;
    if (i > 0 && hits[i - 1].qidx == q) return;
    unsigned long long ct = 0;
    for (uint64_t j = i; j < count && hits[j].qidx == q; ++j) {
        unsigned long long len = hits[j].len;
        if (len + ct > n) {
            len = n - ct;
            hits[j].len = (uint32_t)len;
        }
        ct += len;
        keep[j] = 1;
        if (ct == n) break;
    }
}
__global__ void scatter_kept_kernel(const HitRec* __restrict__ hits, const uint32_t* __restrict__ keep, const uint32_t* __restrict__ pos,
                                    HitRec* __restrict__ out, uint64_t count) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < count && keep[i]) out[pos[i]] = hits[i];
}

int order_and_limit(fmb_results* res, DevBuf<unsigned long long>& keys, uint64_t n_limit, cudaStream_t st) {
    const uint64_t count = res->count;
    if (count == 0) return FMB_OK;
    if (count >= 0xFFFFFFFFull) { set_error("hit-limited search: %llu hits before the limit is applied, split the query batch", (unsigned long long)count); return FMB_EOVERFLOW; }
    const unsigned grid = (unsigned)((count + 255) / 256);
    DevBuf<uint32_t> perm_a, perm_b, qk_a, qk_b;
    DevBuf<unsigned long long> keys_b;
    DevBuf<HitRec> sorted;
    FMB_TRY(perm_a.alloc(count)); FMB_TRY(perm_b.alloc(count)); FMB_TRY(qk_a.alloc(count + 1)); FMB_TRY(qk_b.alloc(count + 1));
    FMB_TRY(keys_b.alloc(count)); FMB_TRY(sorted.alloc(count));
    iota_kernel<<<grid, 256, 0, st>>>(perm_a.p, count);
    size_t tmp_bytes = 0, tmp_bytes2 = 0, tmp_bytes3 = 0;
    FMB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys.p, keys_b.p, perm_a.p, perm_b.p, (int64_t)count, 0, 64, st));
    FMB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes2, qk_a.p, qk_b.p, perm_b.p, perm_a.p, (int64_t)count, 0, 32, st));
    FMB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes3, qk_a.p, qk_b.p, (int64_t)(count + 1), st));
    DevBuf<uint8_t> tmp;
    FMB_TRY(tmp.alloc(std::max(tmp_bytes, std::max(tmp_bytes2, tmp_bytes3))));
    FMB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, keys.p, keys_b.p, perm_a.p, perm_b.p, (int64_t)count, 0, 64, st));     // discovery order ...
    gather_qidx_kernel<<<grid, 256, 0, st>>>(res->hits.p, perm_b.p, qk_a.p, count);
    FMB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes2, qk_a.p, qk_b.p, perm_b.p, perm_a.p, (int64_t)count, 0, 32, st));      // ... within ascending qidx (stable)
    gather_hits_kernel<<<grid, 256, 0, st>>>(res->hits.p, perm_a.p, sorted.p, count);
    // qk_a: keep flags (+ one trailing zero), qk_b: their exclusive sum -- qk_b[count] = number of hits kept
    FMB_CUDA(cudaMemsetAsync(qk_a.p, 0, (count + 1) * sizeof(uint32_t), st));
    limit_rows_kernel<<<grid, 256, 0, st>>>(sorted.p, qk_a.p, count, (unsigned long long)n_limit);
    FMB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes3, qk_a.p, qk_b.p, (int64_t)(count + 1), st));
    scatter_kept_kernel<<<grid, 256, 0, st>>>(sorted.p, qk_a.p, qk_b.p, res->hits.p, count);
    uint32_t kept = 0;
    FMB_CUDA(cudaMemcpyAsync(&kept, qk_b.p + count, sizeof kept, cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    FMB_CUDA(cudaGetLastError());
    note_launches(9);
    res->count = kept;
    res->slots = kept;
    return FMB_OK;
}

// ordered mode: the layout of the discovery-order key (order_key_edge), one slot per error of the search that allows the most
int key_layout(SchemeParams& sp, uint32_t sigma) {
    uint32_t K = 0, total = 0;
    for (uint32_t s = 0; s < sp.n_searches; ++s)
        for (uint32_t p = 0; p < sp.n_parts; ++p) K = std::max<uint32_t>(K, sp.u[s][p]);
    for (uint32_t p = 0; p < sp.n_parts; ++p) total += sp.partition[p];
    sp.key_slots = K;
    sp.key_maxd = total + 2 * K + 2;
    sp.key_ords = 2 * sigma + 2;
    const uint64_t range = (uint64_t)sp.key_maxd + 1 + (uint64_t)sp.key_maxd * sp.key_ords;
    sp.key_bits = 1;
    while ((1ull << sp.key_bits) < range) ++sp.key_bits;
    if (K * sp.key_bits > 56) {
        set_error("hit-limited search: %u errors on %u-symbol queries need %u key bits (56 available)", K, total, K * sp.key_bits);
        return FMB_EUNSUPPORTED;
    }
    return FMB_OK;
}

// The item lists of one search call, `cap` items each.  A pass of the frontier kernel reads one overflow list and fills the other.  In
// text mode it also fills the current text list, which the text kernel of the same pass reads while it appends its text-class
// hand-overs to the other text list: the two swap roles after every text pass.  Edit distance sorts a text list by class first.
struct SchemeLists {
    uint64_t cap = 0;
    DevBuf<Item> ovf[2], text[2], text_sorted;
    DevBuf<unsigned long long> ovf_keys[2];           // ordered mode: the keys of the overflow items
    DevBuf<uint32_t> tkeys[2], tidx[2];
    DevBuf<uint8_t> sort_tmp;
    size_t sort_bytes = 0;

    int alloc(uint64_t items, bool text_mode, bool sort, bool ordered, cudaStream_t st) {
        cap = items;
        for (int b = 0; b < 2; ++b) {
            FMB_TRY(ovf[b].alloc(cap));
            if (text_mode) FMB_TRY(text[b].alloc(cap));
            if (ordered) FMB_TRY(ovf_keys[b].alloc(cap));
        }
        if (sort) {
            FMB_TRY(text_sorted.alloc(cap));
            for (int b = 0; b < 2; ++b) { FMB_TRY(tkeys[b].alloc(cap)); FMB_TRY(tidx[b].alloc(cap)); }
            FMB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, tkeys[0].p, tkeys[1].p, tidx[0].p, tidx[1].p, (int64_t)cap, 0, 10, st));
            FMB_TRY(sort_tmp.alloc(sort_bytes));
        }
        return FMB_OK;
    }
};

// the kernels count what does not fit a list and drop it
int lists_fit(const unsigned long long* h_ctr, uint64_t cap) {
    if (h_ctr[CTR_OVERFLOW] <= cap && h_ctr[CTR_TEXT_A] <= cap && h_ctr[CTR_TEXT_B] <= cap) return FMB_OK;
    set_error("scheme search: frontier lists exceeded %llu items; split the query batch", (unsigned long long)cap);
    return FMB_EOVERFLOW;
}

// The roots [root_base, root_base + roots), pass by pass: the frontier kernel takes the roots (first pass) and the overflow list of the
// previous pass; in text mode the text kernel then decides the single-row items the frontier kernel handed over.  The slab ends when
// every list is empty.  h_ctr: the counter block as the last kernel left it.
int run_slab(const fmb_index* ix, const SchemeParams& sp, const fmb_queries* q, bool ordered, bool pseudo, SchemeLists& L, SchemeOut& so,
             unsigned long long* ctr, unsigned long long* h_ctr, uint64_t root_base, uint64_t roots, cudaStream_t st) {
    static const bool trace = getenv("FMB_TRACE_SCHEME") != nullptr;
    auto read_back = [&]() -> int {
        FMB_CUDA(cudaMemcpyAsync(h_ctr, ctr, CTR_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        FMB_CUDA(cudaStreamSynchronize(st));
        return FMB_OK;
    };
    if (root_base) {                                  // slab level: the previous slab left its lists empty
        FMB_CUDA(cudaMemsetAsync(ctr + CTR_OVERFLOW, 0, 3 * sizeof(unsigned long long), st));   // overflow, roots, text list A
        FMB_CUDA(cudaMemsetAsync(ctr + CTR_TEXT_B, 0, sizeof(unsigned long long), st));
    }
    so.root_base = root_base;
    so.text = L.text[0].p;                            // the text list the frontier kernel fills and the text kernel reads
    so.text_count = ctr + CTR_TEXT_A;
    so.text_next = L.text[1].p;                       // the one the text kernel appends its hand-overs to
    so.text_next_count = ctr + CTR_TEXT_B;
    uint64_t n_in = 0;
    for (int pass = 0;; ++pass) {
        const int cur = pass & 1;                     // the overflow list this pass fills; it reads the other one
        so.overflow = L.ovf[cur].p;
        so.overflow_keys = L.ovf_keys[cur].p;
        so.in_keys = pass ? L.ovf_keys[cur ^ 1].p : nullptr;
        EventPair tr;
        if (trace) cudaEventRecord(tr.a, st);
        if (roots + n_in > 0) FMB_TRY(launch_frontier(ix, sp, q, ordered, pseudo, roots, pass ? L.ovf[cur ^ 1].p : nullptr, n_in, so, st));
        if (trace) cudaEventRecord(tr.b, st);
        FMB_TRY(read_back());
        const size_t ti = so.text_count - ctr, tn = so.text_next_count - ctr;     // counter slots of the two text lists
        if (trace) {
            float ms = 0;
            cudaEventElapsedTime(&ms, tr.a, tr.b);
            fprintf(stderr, "[fmb scheme] slab %llu pass %d frontier kernel: %.3f ms, %llu roots + %llu items in -> %llu text, %llu back, %llu hits so far\n",
                    (unsigned long long)root_base, pass, ms, (unsigned long long)roots, (unsigned long long)n_in, h_ctr[ti], h_ctr[CTR_OVERFLOW], h_ctr[CTR_HITS]);
        }
        FMB_TRY(lists_fit(h_ctr, L.cap));
        if (h_ctr[ti]) {
            // the single-row items of this pass are decided on the text; what survives joins the next text list (a new direction
            // run, a new window) or the overflow list (what must be expanded on the index)
            const unsigned long long n_text = h_ctr[ti], back0 = h_ctr[CTR_OVERFLOW];
            if (trace) cudaEventRecord(tr.a, st);
            const Item* text_in = so.text;
            if (L.text_sorted.p && n_text > 65536) {
                const unsigned grid = (unsigned)((n_text + 255) / 256);
                text_class_keys_kernel<<<grid, 256, 0, st>>>(text_in, n_text, L.tkeys[0].p, L.tidx[0].p);
                FMB_CUDA(cub::DeviceRadixSort::SortPairs(L.sort_tmp.p, L.sort_bytes, L.tkeys[0].p, L.tkeys[1].p, L.tidx[0].p, L.tidx[1].p, (int64_t)n_text, 0, 10, st));
                gather_items_kernel<<<grid, 256, 0, st>>>(text_in, L.tidx[1].p, n_text, L.text_sorted.p);
                FMB_CUDA(cudaGetLastError());
                note_launches(3);
                text_in = L.text_sorted.p;
            }
            FMB_TRY(launch_text(ix, sp, q, text_in, n_text, so, pseudo, st));
            if (trace) cudaEventRecord(tr.b, st);
            FMB_CUDA(cudaMemsetAsync(ctr + ti, 0, sizeof(unsigned long long), st));        // pass level: the text list just read
            FMB_TRY(read_back());
            if (trace) {
                float ms = 0;
                cudaEventElapsedTime(&ms, tr.a, tr.b);
                fprintf(stderr, "[fmb scheme] slab %llu pass %d text kernel: %.3f ms, %llu items -> %llu to the next text list, %llu back\n",
                        (unsigned long long)root_base, pass, ms, n_text, h_ctr[tn], h_ctr[CTR_OVERFLOW] - back0);
            }
            std::swap(so.text, so.text_next);         // the frontier kernel of the next pass appends to what the text kernel began
            std::swap(so.text_count, so.text_next_count);
            FMB_TRY(lists_fit(h_ctr, L.cap));
        }
        if (h_ctr[CTR_OVERFLOW] == 0 && h_ctr[CTR_TEXT_A] == 0 && h_ctr[CTR_TEXT_B] == 0) return FMB_OK;
        // feed the spilled / returned items to the next pass
        n_in = h_ctr[CTR_OVERFLOW];
        roots = 0;
        FMB_CUDA(cudaMemsetAsync(ctr + CTR_OVERFLOW, 0, 2 * sizeof(unsigned long long), st));     // pass level: overflow, roots
        if (pass > 100000) { set_error("scheme search did not terminate"); return FMB_ECUDA; }
    }
}

// n_limit = UINT64_MAX: every hit, in no particular order; else the reference's search_n semantics (SearchNg26.h:408-423)
// pseudo: edit distance without the redundancy filter of search_ng26 (search_pseudo::search<true>, search/SearchPseudo.h:100-165)
int run_scheme(const fmb_index* ix, const fmb_queries* q, const SchemeParams& sp_in, fmb_results** out_res, uint64_t n_limit = UINT64_MAX, bool pseudo = false) {
    SchemeParams sp = sp_in;
    const bool ordered = n_limit != UINT64_MAX;
    if (ordered) FMB_TRY(key_layout(sp, ix->sigma));
    FMB_TRY(set_device(ix->device));
    cudaStream_t st = active_stream(ix);
    auto res = new fmb_results();
    res->device = ix->device;
    res->kind = 0;
    struct Guard { fmb_results* r; ~Guard() { delete r; } } guard{res};

    const uint64_t nq = q->nq;
    const uint64_t n_roots = nq * sp.n_searches;
    // Text mode: the frontier kernel hands single-row items to the text kernel through a global list and gets
    // the survivors back through the overflow list, so the lists scale with the number of roots in flight: the roots are processed
    // in slabs.  Otherwise: all roots at once, the overflow list only takes what the warp stacks cannot hold.
    // (generic layout: Hamming-distance searches stay on the frontier kernel, whose LF^4 jumps absorb mismatches as well as a
    // 4-symbol window does -- measured on the protein workload: 332 M queries/s there against 242 M through the text kernel)
    const bool text_mode = !ordered && (ix->dna || sp.edit) && text_mode_available(ix, q, sp.force_left != 0);
    static const uint64_t env_slab = getenv("FMB_SCHEME_SLAB") ? strtoull(getenv("FMB_SCHEME_SLAB"), nullptr, 10) : 0;
    // (without text mode the roots go in slabs as well: what a slab spills -- warp stacks that ran full -- stays bounded)
    const uint64_t slab = std::min<uint64_t>(std::max<uint64_t>(n_roots, 1), env_slab ? env_slab : (text_mode ? (uint64_t(16) << 20) : (uint64_t(4) << 20)));      // at 30 M roots: 8 M 63.5 ms, 16 M 61.5, 32 M 60.1 (k = 2 edit)
    // small hit limits (n <= 8 rows per query): the kernel keeps the n smallest keys found per query and drops what cannot beat the n-th
    const bool prune_first = ordered && n_limit >= 1 && n_limit <= kMaxPruneN;
    const uint64_t n_best = std::max<uint64_t>(nq, 1) * (prune_first ? n_limit : 1);

    SchemeLists lists;
    // (the class sort is for edit distance only: the Hamming walk has one shape whatever the class)
    FMB_TRY(lists.alloc(std::max<uint64_t>(1u << 20, slab * 2 + (1u << 18)), text_mode, text_mode && sp.edit, ordered, st));
    DevBuf<unsigned long long> best_keys, hit_keys, ctr;
    if (prune_first) FMB_TRY(best_keys.alloc(n_best));
    FMB_TRY(ctr.alloc(CTR_SLOTS));
    EventPair evs;
    double total_ms = 0;
    unsigned long long h_ctr[CTR_SLOTS];
    uint64_t hit_cap = std::max<uint64_t>(1u << 20, nq * 8);
    // (a second attempt runs with the exact size the first one counted; with work-bounding hit limits the count depends on the timing of
    // the pruning, so those retries reserve twice what was counted and may repeat)
    for (int attempt = 0; attempt < (prune_first ? 5 : 2); ++attempt) {
        FMB_TRY(res->hits.alloc(hit_cap));
        if (ordered) FMB_TRY(hit_keys.alloc(hit_cap));
        FMB_CUDA(cudaMemsetAsync(ctr.p, 0, sizeof h_ctr, st));                                   // attempt level: every counter
        SchemeOut so{};
        so.hit_keys = hit_keys.p;
        so.hits = res->hits.p;
        so.hit_count = ctr.p + CTR_HITS;
        so.row_count = ctr.p + CTR_ROWS;
        so.hit_capacity = hit_cap;
        so.overflow_count = ctr.p + CTR_OVERFLOW;
        so.overflow_capacity = lists.cap;
        so.text_capacity = lists.cap;
        so.counters = ctr.p + CTR_EXTENSIONS;
        so.root_counter = ctr.p + CTR_ROOTS;
        so.qidx_base = (uint32_t)q->qidx_base;
        if (prune_first) {
            FMB_CUDA(cudaMemsetAsync(best_keys.p, 0xFF, n_best * sizeof(unsigned long long), st));
            so.best_keys = best_keys.p;
            so.n_queries = nq;
            so.prune_n = (uint32_t)n_limit;
        }
        cudaEventRecord(evs.a, st);
        for (uint64_t root_base = 0; root_base < std::max<uint64_t>(n_roots, 1); root_base += slab) {
            const uint64_t roots = n_roots ? std::min<uint64_t>(slab, n_roots - root_base) : 0;
            FMB_TRY(run_slab(ix, sp, q, ordered, pseudo, lists, so, ctr.p, h_ctr, root_base, roots, st));
        }
        cudaEventRecord(evs.b, st);
        cudaEventSynchronize(evs.b);
        float ms = 0;
        cudaEventElapsedTime(&ms, evs.a, evs.b);
        total_ms += ms;
        if (h_ctr[CTR_HITS] <= hit_cap) break;
        hit_cap = prune_first ? 2 * h_ctr[CTR_HITS] : h_ctr[CTR_HITS];
    }
    if (h_ctr[CTR_HITS] > hit_cap) {
        // (the retries ran with the size counted before: only a hit count that keeps growing between attempts could get here)
        set_error("scheme search: %llu hits do not fit the %llu reserved", h_ctr[CTR_HITS], (unsigned long long)hit_cap);
        return FMB_EOVERFLOW;
    }
    res->count = h_ctr[CTR_HITS];
    res->slots = h_ctr[CTR_HITS];
    res->total_rows = ordered ? UINT64_MAX : h_ctr[CTR_ROWS];      // the hit limit clips intervals afterwards: locate counts again
    res->stats.extensions = h_ctr[CTR_EXTENSIONS];
    res->stats.occ_lookups = h_ctr[CTR_OCC_LOOKUPS];
    res->stats.frontier_peak = h_ctr[CTR_PEAK];
    res->stats.line_requests = h_ctr[CTR_LINE_REQUESTS];
    res->stats.kernel_ms = total_ms;
    res->stats.main_kernel_ms = total_ms;
    if (ordered) FMB_TRY(order_and_limit(res, hit_keys, n_limit, st));
    guard.r = nullptr;
    *out_res = res;
    return FMB_OK;
}

}  // namespace

extern "C" {

static int scheme_entry(const fmb_index* ix, const fmb_queries* q, int edit, uint32_t n_searches, uint32_t n_parts,
                        const uint32_t* pi, const uint32_t* l, const uint32_t* u, const uint32_t* partition, uint64_t n, bool pseudo, fmb_results** out);

int fmb_search_scheme(const fmb_index* ix, const fmb_queries* q, int edit, uint32_t n_searches, uint32_t n_parts,
                      const uint32_t* pi, const uint32_t* l, const uint32_t* u, const uint32_t* partition, fmb_results** out) {
    return fmb_search_scheme_n(ix, q, edit, n_searches, n_parts, pi, l, u, partition, UINT64_MAX, out);
}

int fmb_search_scheme_n(const fmb_index* ix, const fmb_queries* q, int edit, uint32_t n_searches, uint32_t n_parts,
                        const uint32_t* pi, const uint32_t* l, const uint32_t* u, const uint32_t* partition, uint64_t n, fmb_results** out) {
    return scheme_entry(ix, q, edit, n_searches, n_parts, pi, l, u, partition, n, false, out);
}

int fmb_search_scheme_pseudo(const fmb_index* ix, const fmb_queries* q, int edit, uint32_t n_searches, uint32_t n_parts,
                             const uint32_t* pi, const uint32_t* l, const uint32_t* u, const uint32_t* partition, fmb_results** out) {
    return scheme_entry(ix, q, edit, n_searches, n_parts, pi, l, u, partition, UINT64_MAX, true, out);
}

static int scheme_entry(const fmb_index* ix, const fmb_queries* q, int edit, uint32_t n_searches, uint32_t n_parts,
                        const uint32_t* pi, const uint32_t* l, const uint32_t* u, const uint32_t* partition, uint64_t n, bool pseudo, fmb_results** out) {
    if (!ix || !q || !out || !pi || !l || !u || !partition) { set_error("NULL argument"); return FMB_EINVAL; }
    *out = nullptr;
    if (!ix->bidirectional) { set_error("search schemes need a bidirectional index (extendRight)"); return FMB_EINVAL; }
    if (ix->sigma > kMaxSchemeSigma) { set_error("k-error searches support sigma <= %u (index has %u)", kMaxSchemeSigma, ix->sigma); return FMB_EUNSUPPORTED; }
    if (q->device != ix->device) { set_error("queries live on device %d, index on %d", q->device, ix->device); return FMB_EINVAL; }
    if (n_searches == 0 || n_searches > (uint32_t)kMaxSearches || n_parts == 0 || n_parts > (uint32_t)kMaxParts) {
        set_error("scheme shape %u x %u outside [1,%d] x [1,%d]", n_searches, n_parts, kMaxSearches, kMaxParts);
        return FMB_EINVAL;
    }
    SchemeParams sp;
    memset(&sp, 0, sizeof sp);
    sp.n_searches = n_searches;
    sp.n_parts = n_parts;
    sp.edit = edit ? 1 : 0;
    sp.zero_lb_rev = 0;
    uint64_t total = 0;
    for (uint32_t p = 0; p < n_parts; ++p) {
        if (partition[p] == 0 || partition[p] > 0xFFFF) { set_error("partition[%u] = %u out of range", p, partition[p]); return FMB_EINVAL; }
        sp.partition[p] = (uint16_t)partition[p];
        total += partition[p];
    }
    if (total > 0xFFFF) { set_error("query length %llu too long", (unsigned long long)total); return FMB_EINVAL; }
    if (q->nq && (q->min_len != total || q->max_len != total)) {
        set_error("every query must have length sum(partition) = %llu (batch has %u..%u)", (unsigned long long)total, q->min_len, q->max_len);
        return FMB_EINVAL;
    }
    for (uint32_t s = 0; s < n_searches; ++s) {
        uint32_t seen = 0;
        for (uint32_t p = 0; p < n_parts; ++p) {
            uint32_t v = pi[s * n_parts + p];
            if (v >= n_parts || (seen >> v) & 1) { set_error("search %u: pi is not a permutation", s); return FMB_EINVAL; }
            seen |= 1u << v;
            if (l[s * n_parts + p] > kMaxSchemeErrors || u[s * n_parts + p] > kMaxSchemeErrors) { set_error("error bounds above %u are not supported", kMaxSchemeErrors); return FMB_EUNSUPPORTED; }
            sp.pi[s][p] = (uint8_t)v;
            sp.l[s][p] = (uint8_t)l[s * n_parts + p];
            sp.u[s][p] = (uint8_t)u[s * n_parts + p];
        }
        // pi must be connected (each part adjacent to the block searched so far), as every generator produces
        uint32_t lo = sp.pi[s][0], hi = sp.pi[s][0];
        for (uint32_t p = 1; p < n_parts; ++p) {
            uint32_t v = sp.pi[s][p];
            if (v + 1 == lo) lo = v;
            else if (v == hi + 1) hi = v;
            else { set_error("search %u: pi is not a connected order", s); return FMB_EINVAL; }
        }
        uint32_t start = 0;
        for (uint32_t i = 0; i < sp.pi[s][0]; ++i) start += sp.partition[i];
        sp.start[s] = (uint16_t)start;
    }
    if (n == 0) {                                   // search_n_impl returns at once (SearchNg26.h:410)
        auto res = new fmb_results();
        res->device = ix->device;
        res->kind = 0;
        *out = res;
        return FMB_OK;
    }
    return run_scheme(ix, q, sp, out, n, pseudo);
}

int fmb_search_backtracking(const fmb_index* ix, const fmb_queries* q, uint32_t max_errors, fmb_results** out) {
    if (!ix || !q || !out) { set_error("NULL argument"); return FMB_EINVAL; }
    *out = nullptr;
    if (q->device != ix->device) { set_error("queries live on device %d, index on %d", q->device, ix->device); return FMB_EINVAL; }
    if (max_errors > kMaxSchemeErrors) { set_error("error bounds above %u are not supported", kMaxSchemeErrors); return FMB_EUNSUPPORTED; }
    if (ix->sigma > kMaxSchemeSigma) { set_error("k-error searches support sigma <= %u (index has %u)", kMaxSchemeSigma, ix->sigma); return FMB_EUNSUPPORTED; }
    if (q->nq && q->min_len != q->max_len) { set_error("backtracking: all queries of a batch must have the same length"); return FMB_EUNSUPPORTED; }
    if (q->nq && q->max_len == 0) { set_error("backtracking: empty queries"); return FMB_EINVAL; }
    SchemeParams sp;
    memset(&sp, 0, sizeof sp);
    sp.n_searches = 1;
    sp.n_parts = 1;
    sp.edit = 0;
    sp.force_left = 1;
    sp.zero_lb_rev = ix->bidirectional ? 0 : 1;
    sp.partition[0] = (uint16_t)(q->nq ? q->max_len : 1);
    sp.pi[0][0] = 0;
    sp.l[0][0] = 0;
    sp.u[0][0] = (uint8_t)max_errors;
    sp.start[0] = 0;
    return run_scheme(ix, q, sp, out);
}

}  // extern "C"
