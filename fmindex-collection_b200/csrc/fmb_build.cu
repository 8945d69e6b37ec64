// fmb_build.cu -- GPU index construction (SURVEY.md §8f rank 1): suffix sort -> BWT / BWT of the reversed
// text -> text-space sampled suffix array -> device image.  Replaces, for the engine's own use, what the
// reference does with libsais on the CPU (utils.h:97-163, 221-248; fmindex/BiFMIndex.h:64-167).
//
// Suffix sorting = prefix doubling on the device:
//   round 0   key(i) = the first K symbols of suffix i, (symbol+1) packed big-endian, 0 = past the end
//             (so a suffix that is a proper prefix of another sorts first, the order libsais produces);
//             one 64-bit radix sort of (key, i).
//   round r   only suffixes still tied are kept (compacted); they are re-sorted by
//             (group head rank, rank of suffix i + h), h = K * 2^(r-1), and written back in place.
// On random text round 0 leaves ~n^2 / sigma^K ties, so one short extra round finishes; repetitive texts take
// O(log(max LCP / K)) shrinking rounds.  All suffixes of a text are distinct, so the result is unique and the
// BWT is byte-identical to the reference's (tests compare against the oracle).
#include <cub/cub.cuh>

#include "fmb_host.hpp"

namespace fmb {
namespace {

__global__ void reverse_text_kernel(const uint8_t* __restrict__ t, uint64_t n, uint8_t* __restrict__ out) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = t[n - 1 - i];
}

__global__ void check_text_kernel(const uint8_t* __restrict__ t, uint64_t n, uint32_t sigma, uint32_t* bad) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < n && t[i] >= sigma) atomicOr(bad, 1u);
}

__global__ void make_keys_kernel(const uint8_t* __restrict__ t, uint64_t n, uint32_t bits, uint32_t K,
                                 uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t key = 0;
    for (uint32_t j = 0; j < K; ++j) {
        uint64_t v = (i + j < n) ? (uint64_t)t[i + j] + 1 : 0;
        key = (key << bits) | v;
    }
    keys[i] = key;
    vals[i] = (uint32_t)i;
}

// head flag + "position if head" for the max-scan
__global__ void head_flags_kernel(const uint64_t* __restrict__ keys, uint64_t m, uint32_t* __restrict__ headpos) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= m) return;
    bool head = (i == 0) || keys[i] != keys[i - 1];
    headpos[i] = head ? (uint32_t)i : 0u;
}

struct MaxOp {
    __host__ __device__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};

// round 0: ISA[sa[i]] = head(i); tied flag = group larger than one
__global__ void assign_ranks0_kernel(const uint32_t* __restrict__ sa, const uint32_t* __restrict__ head, uint64_t n,
                                     uint32_t* __restrict__ isa, uint8_t* __restrict__ tied) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t h = head[i];
    isa[sa[i]] = h;
    bool single = (h == i) && (i + 1 == n || head[i + 1] == i + 1);
    tied[i] = single ? 0 : 1;
}

struct IsTied {
    const uint8_t* tied;
    __host__ __device__ bool operator()(uint32_t i) const { return tied[i] != 0; }
};

// later rounds: key = (head rank << 32) | (rank of suffix + h, +1; 0 past the end)
__global__ void make_keys_round_kernel(const uint32_t* __restrict__ P, const uint32_t* __restrict__ Hd,
                                       const uint32_t* __restrict__ sa, const uint32_t* __restrict__ isa, uint64_t n,
                                       uint64_t h, uint64_t m, uint64_t* __restrict__ keys, uint32_t* __restrict__ suf) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j >= m) return;
    uint32_t s = sa[P[j]];
    uint64_t nx = (uint64_t)s + h;
    uint64_t r = nx < n ? (uint64_t)isa[nx] + 1 : 0;
    keys[j] = ((uint64_t)Hd[j] << 32) | r;
    suf[j] = s;
}

// write back one refinement round; headidx[j] = index (within the tied list) of the head of j's new group
__global__ void write_back_kernel(const uint32_t* __restrict__ P, const uint32_t* __restrict__ suf_sorted,
                                  const uint32_t* __restrict__ headidx, uint64_t m, uint32_t* __restrict__ sa,
                                  uint32_t* __restrict__ isa, uint32_t* __restrict__ Hd_new, uint8_t* __restrict__ tied) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j >= m) return;
    uint32_t hj = headidx[j];
    uint32_t rank = P[hj];
    uint32_t s = suf_sorted[j];
    sa[P[j]] = s;
    isa[s] = rank;
    Hd_new[j] = rank;
    bool single = (hj == j) && (j + 1 == m || headidx[j + 1] == j + 1);
    tied[j] = single ? 0 : 1;
}

__global__ void gather_u32_kernel(const uint32_t* __restrict__ src, const uint32_t* __restrict__ idx, uint64_t m, uint32_t* __restrict__ out) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j < m) out[j] = src[idx[j]];
}

__global__ void bwt_from_sa_kernel(const uint8_t* __restrict__ t, const uint32_t* __restrict__ sa, uint64_t n, uint8_t* __restrict__ bwt) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t p = sa[i];
    bwt[i] = t[p ? p - 1 : n - 1];        // utils.h:145-163: T[(SA[i] + n - 1) % n]
}

struct IsDelim {
    const uint8_t* t;
    __host__ __device__ bool operator()(uint32_t i) const { return t[i] == 0; }
};

// (seqId, pos) of text position p: delims = sorted text positions holding 0       (BiFMIndex.h:121-135)
__device__ __forceinline__ void seq_pos(const uint32_t* __restrict__ delims, uint32_t nd, uint32_t p, uint32_t& seq, uint32_t& pos) {
    uint32_t lo = 0, hi = nd;             // first delimiter position >= p  ->  number of delimiters < p
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(delims + mid) < p) lo = mid + 1; else hi = mid;
    }
    seq = lo;
    pos = p - (lo ? __ldg(delims + lo - 1) + 1 : 0);
}

// one thread per 64 rows: marker word + number of samples in it
__global__ void sample_words_kernel(const uint32_t* __restrict__ sa, uint64_t n, const uint32_t* __restrict__ delims, uint32_t nd,
                                    uint32_t rate, uint64_t words, uint64_t* __restrict__ bitmap, uint32_t* __restrict__ cnt) {
    uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (w > words) return;
    if (w == words) { cnt[w] = 0; return; }
    uint64_t bits = 0;
    for (uint32_t r = 0; r < 64; ++r) {
        uint64_t i = w * 64 + r;
        if (i >= n) break;
        uint32_t seq, pos;
        seq_pos(delims, nd, sa[i], seq, pos);
        if (pos % rate == 0) bits |= uint64_t(1) << r;
    }
    bitmap[w] = bits;
    cnt[w] = __popcll(bits);
}
__global__ void sample_fill_kernel(const uint32_t* __restrict__ sa, uint64_t n, const uint32_t* __restrict__ delims, uint32_t nd,
                                   uint64_t words, const uint64_t* __restrict__ bitmap, const uint32_t* __restrict__ before,
                                   uint4* __restrict__ marks, uint2* __restrict__ samples) {
    uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (w >= words) return;
    uint64_t bits = bitmap[w];
    uint32_t k = before[w];
    marks[w] = make_uint4((uint32_t)bits, (uint32_t)(bits >> 32), k, 0);
    while (bits) {
        uint32_t r = __ffsll((long long)bits) - 1;
        bits &= bits - 1;
        uint32_t seq, pos;
        seq_pos(delims, nd, sa[w * 64 + r], seq, pos);
        samples[k++] = make_uint2(seq, pos);
    }
}

template <typename T>
int scan_max_inclusive(const T* in, T* out, uint64_t m, cudaStream_t st) {
    size_t tmp_bytes = 0;
    FMB_CUDA(cub::DeviceScan::InclusiveScan(nullptr, tmp_bytes, in, out, MaxOp{}, (int64_t)m, st));
    DevBuf<uint8_t> tmp;
    FMB_TRY(tmp.alloc(tmp_bytes));
    FMB_CUDA(cub::DeviceScan::InclusiveScan(tmp.p, tmp_bytes, in, out, MaxOp{}, (int64_t)m, st));
    return FMB_OK;
}

int sort_pairs(uint64_t* k_in, uint64_t* k_out, uint32_t* v_in, uint32_t* v_out, uint64_t m, int end_bit, cudaStream_t st) {
    size_t tmp_bytes = 0;
    FMB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in, k_out, v_in, v_out, (int64_t)m, 0, end_bit, st));
    DevBuf<uint8_t> tmp;
    FMB_TRY(tmp.alloc(tmp_bytes));
    FMB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, k_in, k_out, v_in, v_out, (int64_t)m, 0, end_bit, st));
    return FMB_OK;
}

template <typename Pred>
int select_positions(uint64_t count, Pred pred, uint32_t* out, uint64_t* n_selected, cudaStream_t st) {
    cub::CountingInputIterator<uint32_t> it(0);
    DevBuf<uint64_t> d_num;
    FMB_TRY(d_num.alloc(1));
    size_t tmp_bytes = 0;
    FMB_CUDA(cub::DeviceSelect::If(nullptr, tmp_bytes, it, out, d_num.p, (int64_t)count, pred, st));
    DevBuf<uint8_t> tmp;
    FMB_TRY(tmp.alloc(tmp_bytes));
    FMB_CUDA(cub::DeviceSelect::If(tmp.p, tmp_bytes, it, out, d_num.p, (int64_t)count, pred, st));
    FMB_CUDA(cudaMemcpyAsync(n_selected, d_num.p, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    FMB_CUDA(cudaStreamSynchronize(st));
    return FMB_OK;
}

struct FlagSet {
    const uint8_t* f;
    __host__ __device__ bool operator()(uint32_t i) const { return f[i] != 0; }
};

// suffix array of d_text[0,n) into sa (device, n entries)
int suffix_sort(const uint8_t* d_text, uint64_t n, uint32_t sigma, DevBuf<uint32_t>& sa, cudaStream_t st, int* rounds_out) {
    uint32_t bits = 1;
    while ((1u << bits) < sigma + 1) ++bits;
    const uint32_t K = 64 / bits;
    FMB_TRY(sa.alloc(n));
    DevBuf<uint32_t> isa, P, Hd;
    DevBuf<uint8_t> tied;
    FMB_TRY(isa.alloc(n));
    FMB_TRY(tied.alloc(n));
    uint64_t m = 0;
    {
        DevBuf<uint64_t> k0, k1;
        DevBuf<uint32_t> v0, head;
        FMB_TRY(k0.alloc(n));
        FMB_TRY(k1.alloc(n));
        FMB_TRY(v0.alloc(n));
        make_keys_kernel<<<grid_for(n, 256), 256, 0, st>>>(d_text, n, bits, K, k0.p, v0.p);
        FMB_CUDA(cudaGetLastError());
        FMB_TRY(sort_pairs(k0.p, k1.p, v0.p, sa.p, n, (int)(bits * K), st));
        k0.release();
        v0.release();
        FMB_TRY(head.alloc(n));
        head_flags_kernel<<<grid_for(n, 256), 256, 0, st>>>(k1.p, n, head.p);
        FMB_CUDA(cudaGetLastError());
        FMB_TRY(scan_max_inclusive(head.p, head.p, n, st));
        k1.release();
        assign_ranks0_kernel<<<grid_for(n, 256), 256, 0, st>>>(sa.p, head.p, n, isa.p, tied.p);
        FMB_CUDA(cudaGetLastError());
        // compact the tied rows
        FMB_TRY(P.alloc(n));
        FMB_TRY(select_positions(n, FlagSet{tied.p}, P.p, &m, st));
        if (m) {
            DevBuf<uint32_t> Pm, Hm;
            FMB_TRY(Pm.alloc(m));
            FMB_TRY(Hm.alloc(m));
            FMB_CUDA(cudaMemcpyAsync(Pm.p, P.p, m * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
            gather_u32_kernel<<<grid_for(m, 256), 256, 0, st>>>(head.p, Pm.p, m, Hm.p);
            FMB_CUDA(cudaGetLastError());
            FMB_CUDA(cudaStreamSynchronize(st));
            P = std::move(Pm);
            Hd = std::move(Hm);
        } else {
            P.release();
        }
    }
    tied.release();
    int rounds = 0;
    uint64_t h = K;
    while (m) {
        ++rounds;
        if (rounds > 64) { set_error("suffix sort did not converge"); return FMB_ECUDA; }
        DevBuf<uint64_t> k0, k1;
        DevBuf<uint32_t> s0, s1, hidx, Hn;
        DevBuf<uint8_t> t2;
        FMB_TRY(k0.alloc(m)); FMB_TRY(k1.alloc(m)); FMB_TRY(s0.alloc(m)); FMB_TRY(s1.alloc(m));
        FMB_TRY(hidx.alloc(m)); FMB_TRY(Hn.alloc(m)); FMB_TRY(t2.alloc(m));
        make_keys_round_kernel<<<grid_for(m, 256), 256, 0, st>>>(P.p, Hd.p, sa.p, isa.p, n, h, m, k0.p, s0.p);
        FMB_CUDA(cudaGetLastError());
        FMB_TRY(sort_pairs(k0.p, k1.p, s0.p, s1.p, m, 64, st));
        head_flags_kernel<<<grid_for(m, 256), 256, 0, st>>>(k1.p, m, hidx.p);
        FMB_CUDA(cudaGetLastError());
        FMB_TRY(scan_max_inclusive(hidx.p, hidx.p, m, st));
        write_back_kernel<<<grid_for(m, 256), 256, 0, st>>>(P.p, s1.p, hidx.p, m, sa.p, isa.p, Hn.p, t2.p);
        FMB_CUDA(cudaGetLastError());
        // compact (P, Hn) by the new tied flags
        DevBuf<uint32_t> sel;
        FMB_TRY(sel.alloc(m));
        uint64_t m2 = 0;
        FMB_TRY(select_positions(m, FlagSet{t2.p}, sel.p, &m2, st));
        if (m2) {
            DevBuf<uint32_t> P2, H2;
            FMB_TRY(P2.alloc(m2));
            FMB_TRY(H2.alloc(m2));
            gather_u32_kernel<<<grid_for(m2, 256), 256, 0, st>>>(P.p, sel.p, m2, P2.p);
            gather_u32_kernel<<<grid_for(m2, 256), 256, 0, st>>>(Hn.p, sel.p, m2, H2.p);
            FMB_CUDA(cudaGetLastError());
            FMB_CUDA(cudaStreamSynchronize(st));
            P = std::move(P2);
            Hd = std::move(H2);
        }
        m = m2;
        h *= 2;
    }
    FMB_CUDA(cudaStreamSynchronize(st));
    if (rounds_out) *rounds_out = rounds;
    return FMB_OK;
}

}  // namespace
}  // namespace fmb

using namespace fmb;

extern "C" int fmb_index_build(fmb_index** out, int device, uint32_t sigma, const uint8_t* text, uint64_t n,
                               uint32_t sampling_rate, int bidirectional, int text_on_device) {
    if (!text) { set_error("text is NULL"); return FMB_EINVAL; }
    if (sampling_rate == 0) { set_error("sampling_rate must be >= 1"); return FMB_EINVAL; }
    fmb_index* ix = nullptr;
    FMB_TRY(new_index(&ix, device, sigma, n, bidirectional != 0, 0));
    ix->allowed_tables = plan_tables(ix, n / sampling_rate + 1);
    struct Guard {
        fmb_index* ix;
        ~Guard() { if (ix) fmb_index_destroy(ix); }
    } guard{ix};
    cudaStream_t st = ix->stream;
    DevBuf<uint8_t> own_text;
    const uint8_t* d_text = text;
    if (!text_on_device) {
        FMB_TRY(own_text.alloc(n));
        FMB_CUDA(cudaMemcpyAsync(own_text.p, text, n, cudaMemcpyHostToDevice, st));
        d_text = own_text.p;
    }
    {
        DevBuf<uint32_t> bad;
        FMB_TRY(bad.alloc(1));
        FMB_CUDA(cudaMemsetAsync(bad.p, 0, 4, st));
        check_text_kernel<<<grid_for(n, 256), 256, 0, st>>>(d_text, n, sigma, bad.p);
        uint32_t h_bad = 0;
        FMB_CUDA(cudaMemcpyAsync(&h_bad, bad.p, 4, cudaMemcpyDeviceToHost, st));
        FMB_CUDA(cudaStreamSynchronize(st));
        if (h_bad) { set_error("text contains a symbol >= sigma (%u)", sigma); return FMB_EINVAL; }
    }
    DevBuf<uint8_t> bwt;
    FMB_TRY(bwt.alloc(n));
    {
        // forward direction: SA -> BWT -> samples
        DevBuf<uint32_t> sa;
        int rounds = 0;
        FMB_TRY(suffix_sort(d_text, n, sigma, sa, st, &rounds));
        bwt_from_sa_kernel<<<grid_for(n, 256), 256, 0, st>>>(d_text, sa.p, n, bwt.p);
        FMB_CUDA(cudaGetLastError());
        // delimiter text positions
        DevBuf<uint32_t> delims;
        FMB_TRY(delims.alloc(n));
        uint64_t nd = 0;
        FMB_TRY(select_positions(n, IsDelim{d_text}, delims.p, &nd, st));
        const uint64_t words = n / 64 + 1;
        DevBuf<uint64_t> bitmap;
        DevBuf<uint32_t> cnt;
        FMB_TRY(bitmap.alloc(words));
        FMB_TRY(cnt.alloc(words + 1));
        sample_words_kernel<<<grid_for(words + 1, 128), 128, 0, st>>>(sa.p, n, delims.p, (uint32_t)nd, sampling_rate, words, bitmap.p, cnt.p);
        FMB_CUDA(cudaGetLastError());
        FMB_TRY(exclusive_sum_u32(cnt.p, cnt.p, words + 1, st));
        uint32_t ns = 0;
        FMB_CUDA(cudaMemcpyAsync(&ns, cnt.p + words, 4, cudaMemcpyDeviceToHost, st));
        FMB_CUDA(cudaStreamSynchronize(st));
        FMB_TRY(ix->marks.alloc(words));
        FMB_TRY(ix->samples.alloc(ns));
        sample_fill_kernel<<<grid_for(words, 128), 128, 0, st>>>(sa.p, n, delims.p, (uint32_t)nd, words, bitmap.p, cnt.p, ix->marks.p, ix->samples.p);
        FMB_CUDA(cudaGetLastError());
        FMB_CUDA(cudaStreamSynchronize(st));
        ix->n_samples = ns;
    }
    FMB_TRY(build_occ_from_device_bwt(ix, 0, bwt.p));
    if (bidirectional) {
        DevBuf<uint8_t> rev;
        FMB_TRY(rev.alloc(n));
        reverse_text_kernel<<<grid_for(n, 256), 256, 0, st>>>(d_text, n, rev.p);
        FMB_CUDA(cudaGetLastError());
        own_text.release();                 // the forward text is no longer needed (no-op for caller-owned text)
        DevBuf<uint32_t> sa;
        FMB_TRY(suffix_sort(rev.p, n, sigma, sa, st, nullptr));
        bwt_from_sa_kernel<<<grid_for(n, 256), 256, 0, st>>>(rev.p, sa.p, n, bwt.p);
        FMB_CUDA(cudaGetLastError());
        sa.release();
        rev.release();
        FMB_TRY(build_occ_from_device_bwt(ix, 1, bwt.p));
    }
    bwt.release();
    FMB_TRY(compute_C(ix));
    FMB_TRY(build_search_tables(ix));
    FMB_TRY(build_locate_tables(ix));
    guard.ix = nullptr;
    *out = ix;
    pool_trim();
    return FMB_OK;
}
