"""ctypes binding of include/fmb200.h.  Mirrors the C-ABI one to one; numpy arrays in, numpy arrays out."""
import ctypes as C
import os

import numpy as np

from . import build as _build

_LIB = None

HIT_DTYPE = np.dtype([("qidx", "<u8"), ("lb", "<u8"), ("lb_rev", "<u8"), ("len", "<u8"), ("steps", "<u8"), ("e", "<u8")])
LOC_DTYPE = np.dtype([("qidx", "<u8"), ("seq", "<u8"), ("pos", "<u8"), ("e", "<u8")])
LOC32_DTYPE = np.dtype([("qidx", "<u4"), ("seq", "<u4"), ("pos", "<u4"), ("e", "<u4")])
SMEM_DTYPE = np.dtype([("qidx", "<u8"), ("begin", "<u8"), ("end", "<u8"), ("lb", "<u8"), ("len", "<u8")])
SMEM_LOC_DTYPE = np.dtype([("qidx", "<u8"), ("begin", "<u8"), ("end", "<u8"), ("seq", "<u8"), ("pos", "<u8")])
UINT64_MAX = (1 << 64) - 1


class IndexInfo(C.Structure):
    _fields_ = [("n", C.c_uint64), ("sigma", C.c_uint32), ("bidirectional", C.c_uint32), ("n_samples", C.c_uint64),
                ("n_delims", C.c_uint64), ("device_bytes", C.c_uint64), ("occ_block_bytes", C.c_uint32),
                ("occ_block_rows", C.c_uint32), ("device", C.c_int32), ("tables", C.c_uint32), ("flags", C.c_uint32),
                ("text_tables", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("extensions", C.c_uint64), ("occ_lookups", C.c_uint64), ("lf_steps", C.c_uint64),
                ("frontier_peak", C.c_uint64), ("kernel_ms", C.c_double), ("main_kernel_ms", C.c_double),
                ("line_requests", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]


class FmbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"fmb200 error {code}: {msg}")
        self.code = code


def lib_path():
    return _build.LIB


# every symbol include/fmb200.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "fmb_last_error", "fmb_device_count", "fmb_version",
    "fmb_index_create", "fmb_index_create_ex", "fmb_index_build", "fmb_index_destroy", "fmb_index_get_info", "fmb_index_get_C", "fmb_index_export", "fmb_index_export_blocks",
    "fmb_string_symbol", "fmb_string_rank", "fmb_string_prefix_rank", "fmb_string_all_ranks",
    "fmb_cursor_extend", "fmb_cursor_extend_all",
    "fmb_queries_upload", "fmb_queries_upload_revcomp", "fmb_queries_upload_packed", "fmb_pack_symbols", "fmb_queries_destroy", "fmb_queries_count",
    "fmb_search_exact", "fmb_search_scheme", "fmb_search_scheme_n", "fmb_search_scheme_pseudo", "fmb_search_backtracking", "fmb_locate", "fmb_locate_rows", "fmb_sample_value",
    "fmb_search_smems", "fmb_locate_smems", "fmb_results_fetch_smems", "fmb_results_fetch_smem_locs",
    "fmb_results_count", "fmb_results_kind", "fmb_results_fetch_hits", "fmb_results_fetch_locs", "fmb_results_fetch_locs32",
    "fmb_results_get_stats", "fmb_results_destroy",
    "fmb_search_and_locate", "fmb_search_and_locate_packed", "fmb_search_and_locate_multi", "fmb_search_and_locate_parts", "fmb_index_replicate", "fmb_index_save", "fmb_index_load", "fmb_checksum64",
    "fmb_index_sequence_count", "fmb_index_sequence_lengths", "fmb_extract", "fmb_index_reconstruct_text",
    "fmb_index_set_exact_mode", "fmb_index_set_locate_mode", "fmb_synth_text_device", "fmb_synth_reads_device", "fmb_synth_reads_err_device", "fmb_synth_repeat_text_device", "fmb_synth_unit_reads_device", "fmb_index_set_stream", "fmb_set_image_budget", "fmb_measure_gather", "fmb_kernel_launch_count", "fmb_device_free", "fmb_copy_to_host", "fmb_host_alloc_pinned", "fmb_host_free_pinned",
]


def lib():
    """Load libfmb200.so (building it first if sources are newer).  Raises if it cannot be loaded: the product
    path has no fallback."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.build()
    if not os.path.exists(path):
        raise FmbError(-2, f"{path} missing: the CUDA extension is required")
    L = C.CDLL(path)
    L.fmb_last_error.restype = C.c_char_p
    L.fmb_version.restype = C.c_char_p
    L.fmb_results_count.restype = C.c_uint64
    L.fmb_queries_count.restype = C.c_uint64
    L.fmb_kernel_launch_count.restype = C.c_uint64
    L.fmb_checksum64.restype = C.c_uint64
    L.fmb_checksum64.argtypes = [C.c_void_p, C.c_uint64]
    L.fmb_host_alloc_pinned.restype = C.c_void_p
    L.fmb_host_alloc_pinned.argtypes = [C.c_uint64]
    L.fmb_host_free_pinned.argtypes = [C.c_void_p]
    for name in ("fmb_results_count", "fmb_results_kind", "fmb_results_destroy", "fmb_queries_destroy",
                 "fmb_queries_count", "fmb_index_destroy"):
        getattr(L, name).argtypes = [C.c_void_p]
    _LIB = L
    return L


def _check(rc):
    if rc != 0:
        raise FmbError(rc, lib().fmb_last_error().decode())


def device_count():
    return lib().fmb_device_count()


def _ptr(a, typ=C.c_void_p):
    if a is None:
        return typ()
    return a.ctypes.data_as(typ)


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def _u64(a):
    return np.ascontiguousarray(a, dtype=np.uint64)


class Index:
    """Device image of a BiFMIndex / FMIndex (fmindex/BiFMIndex.h, fmindex/FMIndex.h of the reference)."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def from_bwt(cls, sigma, bwt, bwt_rev, sample_bitmap, sample_seq, sample_pos, device=0, no_delim=False, reuse_rev=False):
        """no_delim / reuse_rev: the BiFMIndex::NoDelim / ::ReuseRev variants of the reference (FMB_INDEX_* flags)"""
        bwt = _u8(bwt)
        bwt_rev = None if bwt_rev is None else _u8(bwt_rev)
        bm, sq, sp = _u64(sample_bitmap), _u32(sample_seq), _u32(sample_pos)
        h = C.c_void_p()
        _check(lib().fmb_index_create_ex(C.byref(h), C.c_int(device), C.c_uint32(sigma), C.c_uint64(bwt.size), _ptr(bwt),
                                         _ptr(bwt_rev), _ptr(bm), _ptr(sq), _ptr(sp), C.c_uint64(sq.size),
                                         C.c_uint32((1 if no_delim else 0) | (2 if reuse_rev else 0))))
        return cls(h)

    @classmethod
    def load(cls, path, device=0):
        """loadIndex (fmindex/diskStorage.h:20-27): read the flat index file written by save() and rebuild the device tables"""
        h = C.c_void_p()
        _check(lib().fmb_index_load(C.byref(h), C.c_int(device), os.fsencode(path)))
        return cls(h)

    def save(self, path):
        """saveIndex (fmindex/diskStorage.h:13-18)"""
        _check(lib().fmb_index_save(self.h, os.fsencode(path)))

    @classmethod
    def build(cls, sigma, text, sampling_rate=16, bidirectional=True, device=0):
        """GPU construction from the concatenated text s0 0 s1 0 ... (numpy uint8 on the host)."""
        text = _u8(text)
        h = C.c_void_p()
        _check(lib().fmb_index_build(C.byref(h), C.c_int(device), C.c_uint32(sigma), _ptr(text), C.c_uint64(text.size),
                                     C.c_uint32(sampling_rate), C.c_int(1 if bidirectional else 0), C.c_int(0)))
        return cls(h)

    @classmethod
    def build_from_device_text(cls, sigma, d_text_ptr, n, sampling_rate=16, bidirectional=True, device=0):
        h = C.c_void_p()
        _check(lib().fmb_index_build(C.byref(h), C.c_int(device), C.c_uint32(sigma), C.c_void_p(d_text_ptr), C.c_uint64(n),
                                     C.c_uint32(sampling_rate), C.c_int(1 if bidirectional else 0), C.c_int(1)))
        return cls(h)

    def replicate(self, device):
        """a replica of the finished device image on another GPU (peer-to-peer copy, no rebuild)"""
        h = C.c_void_p()
        _check(lib().fmb_index_replicate(self.h, C.c_int(device), C.byref(h)))
        return Index(h)

    def close(self):
        if self.h:
            lib().fmb_index_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def info(self):
        i = IndexInfo()
        _check(lib().fmb_index_get_info(self.h, C.byref(i)))
        return i

    @property
    def C(self):
        out = np.zeros(self.info.sigma + 1, dtype=np.uint64)
        _check(lib().fmb_index_get_C(self.h, _ptr(out)))
        return out

    def export(self):
        i = self.info
        bwt = np.zeros(i.n, dtype=np.uint8)
        rev = np.zeros(i.n, dtype=np.uint8) if i.bidirectional else None
        bm = np.zeros((i.n + 63) // 64, dtype=np.uint64)
        sq = np.zeros(i.n_samples, dtype=np.uint32)
        sp = np.zeros(i.n_samples, dtype=np.uint32)
        _check(lib().fmb_index_export(self.h, _ptr(bwt), _ptr(rev), _ptr(bm), _ptr(sq), _ptr(sp)))
        return bwt, rev, bm, sq, sp

    def export_blocks(self, dir=0):
        """raw bytes of the one-symbol occurrence table (the blocks the kernels read) and the bytes per 64-row block"""
        nbytes, stride = C.c_uint64(0), C.c_uint32(0)
        _check(lib().fmb_index_export_blocks(self.h, C.c_int(dir), None, C.c_uint64(0), C.byref(nbytes), C.byref(stride)))
        out = np.zeros(nbytes.value, dtype=np.uint8)
        _check(lib().fmb_index_export_blocks(self.h, C.c_int(dir), _ptr(out), C.c_uint64(out.size), C.byref(nbytes), C.byref(stride)))
        return out, stride.value

    def set_exact_mode(self, mode):
        """0 = auto (two-symbol steps when available), 1 = one-symbol kernel (fills the algorithmic counters), 2 = two-symbol"""
        _check(lib().fmb_index_set_exact_mode(self.h, C.c_int(mode)))

    def set_locate_mode(self, mode):
        """0 = auto (locate shortcut table when available), 1 = always walk LF steps to the nearest sample"""
        _check(lib().fmb_index_set_locate_mode(self.h, C.c_int(mode)))

    # String_c
    def symbol(self, idx, dir=0):
        idx = _u64(idx)
        out = np.zeros(idx.size, dtype=np.uint8)
        _check(lib().fmb_string_symbol(self.h, C.c_int(dir), _ptr(idx), C.c_uint64(idx.size), _ptr(out)))
        return out

    def rank(self, idx, symb, dir=0):
        idx, symb = _u64(idx), _u8(symb)
        out = np.zeros(idx.size, dtype=np.uint64)
        _check(lib().fmb_string_rank(self.h, C.c_int(dir), _ptr(idx), _ptr(symb), C.c_uint64(idx.size), _ptr(out)))
        return out

    def prefix_rank(self, idx, symb, dir=0):
        idx, symb = _u64(idx), _u8(symb)
        out = np.zeros(idx.size, dtype=np.uint64)
        _check(lib().fmb_string_prefix_rank(self.h, C.c_int(dir), _ptr(idx), _ptr(symb), C.c_uint64(idx.size), _ptr(out)))
        return out

    def all_ranks(self, idx, dir=0):
        idx = _u64(idx)
        s = self.info.sigma
        rs = np.zeros((idx.size, s), dtype=np.uint64)
        prs = np.zeros((idx.size, s), dtype=np.uint64)
        _check(lib().fmb_string_all_ranks(self.h, C.c_int(dir), _ptr(idx), C.c_uint64(idx.size), _ptr(rs), _ptr(prs)))
        return rs, prs

    # cursors: arrays of shape (count, 4) = lb, lbRev, len, steps
    def extend(self, cur, symb, right):
        cur, symb = _u64(cur).reshape(-1, 4), _u8(symb)
        out = np.zeros_like(cur)
        _check(lib().fmb_cursor_extend(self.h, C.c_int(right), _ptr(cur), _ptr(symb), C.c_uint64(cur.shape[0]), _ptr(out)))
        return out

    def extend_all(self, cur, right):
        cur = _u64(cur).reshape(-1, 4)
        out = np.zeros((cur.shape[0], self.info.sigma, 4), dtype=np.uint64)
        _check(lib().fmb_cursor_extend_all(self.h, C.c_int(right), _ptr(cur), C.c_uint64(cur.shape[0]), _ptr(out)))
        return out

    # searches
    def upload(self, symbols, offsets, complement=None, packed=None):
        """complement: table of sigma symbols (DNA: [0, 4, 3, 2, 1]) -> the device batch holds every query followed by its reverse
        complement (2 nq queries, example/utils.h:62-74), built on the device.  packed = pack_queries(symbols): the 2-bit host form"""
        return Queries(self, symbols, offsets, complement, packed)

    def search_exact(self, queries):
        r = C.c_void_p()
        _check(lib().fmb_search_exact(self.h, queries.h, C.byref(r)))
        return Results(r)

    def search_scheme(self, queries, scheme, partition, edit, n=None):
        """n = hit limit per query in rows (search_n, SearchNg26.h:408-423): hits come back in (qidx, discovery) order"""
        pi, l, u = (np.ascontiguousarray(a, dtype=np.uint32) for a in scheme)
        part = _u32(partition)
        r = C.c_void_p()
        if n is None:
            _check(lib().fmb_search_scheme(self.h, queries.h, C.c_int(1 if edit else 0), C.c_uint32(pi.shape[0]),
                                           C.c_uint32(pi.shape[1]), _ptr(pi), _ptr(l), _ptr(u), _ptr(part), C.byref(r)))
        else:
            _check(lib().fmb_search_scheme_n(self.h, queries.h, C.c_int(1 if edit else 0), C.c_uint32(pi.shape[0]),
                                             C.c_uint32(pi.shape[1]), _ptr(pi), _ptr(l), _ptr(u), _ptr(part), C.c_uint64(n), C.byref(r)))
        return Results(r)

    def search_scheme_pseudo(self, queries, scheme, partition, edit):
        """search_pseudo::search<Edit> on the part form of an expanded scheme: edit distance without redundancy filter"""
        pi, l, u = (np.ascontiguousarray(a, dtype=np.uint32) for a in scheme)
        part = _u32(partition)
        r = C.c_void_p()
        _check(lib().fmb_search_scheme_pseudo(self.h, queries.h, C.c_int(1 if edit else 0), C.c_uint32(pi.shape[0]),
                                              C.c_uint32(pi.shape[1]), _ptr(pi), _ptr(l), _ptr(u), _ptr(part), C.byref(r)))
        return Results(r)

    def search_backtracking(self, queries, max_errors):
        r = C.c_void_p()
        _check(lib().fmb_search_backtracking(self.h, queries.h, C.c_uint32(max_errors), C.byref(r)))
        return Results(r)

    def locate(self, hits):
        r = C.c_void_p()
        _check(lib().fmb_locate(self.h, hits.h, C.byref(r)))
        return Results(r)

    def search_smems(self, queries, min_len=1):
        """super-maximal exact matches of every query (fmb_search_smems): the stretches of a query that occur in one sequence of the
        collection and cannot be extended on either side, at least min_len symbols long, ordered by qidx, then begin"""
        r = C.c_void_p()
        _check(lib().fmb_search_smems(self.h, queries.h, C.c_uint32(min_len), C.byref(r)))
        return Results(r)

    def locate_smems(self, results, max_occ=None):
        """the first min(len, max_occ) rows of every SMEM's interval, located (fmb_locate_smems; max_occ None: every row)"""
        r = C.c_void_p()
        _check(lib().fmb_locate_smems(self.h, results.h, C.c_uint64(UINT64_MAX if max_occ is None else int(max_occ)), C.byref(r)))
        return Results(r)

    def locate_rows(self, rows):
        """index.locate(row) for many rows: (seq, pos, steps) arrays"""
        rows = _u64(rows)
        seq = np.zeros(rows.size, dtype=np.uint32)
        pos = np.zeros(rows.size, dtype=np.uint32)
        steps = np.zeros(rows.size, dtype=np.uint64)
        _check(lib().fmb_locate_rows(self.h, _ptr(rows), C.c_uint64(rows.size), _ptr(seq), _ptr(pos), _ptr(steps)))
        return seq, pos, steps

    def sample_value(self, rows):
        """index.single_locate_step(row) for many rows: (has, seq, pos) arrays"""
        rows = _u64(rows)
        has = np.zeros(rows.size, dtype=np.uint8)
        seq = np.zeros(rows.size, dtype=np.uint32)
        pos = np.zeros(rows.size, dtype=np.uint32)
        _check(lib().fmb_sample_value(self.h, _ptr(rows), C.c_uint64(rows.size), _ptr(has), _ptr(seq), _ptr(pos)))
        return has, seq, pos

    def sequence_count(self):
        """number of sequences of the collection (= delimiters)"""
        c = C.c_uint64()
        _check(lib().fmb_index_sequence_count(self.h, C.byref(c)))
        return c.value

    def sequence_lengths(self):
        """symbols per sequence, delimiter excluded (uint64 array)"""
        out = np.zeros(self.sequence_count(), dtype=np.uint64)
        _check(lib().fmb_index_sequence_lengths(self.h, _ptr(out)))
        return out

    def extract(self, seq, begin, end, with_stats=False):
        """text of sequence seq[i] at [begin[i], end[i]) for every i, read back from the index on the GPU (fmb_extract).  Scalars give
        one uint8 array; arrays give a list of uint8 arrays (views of one buffer).  with_stats=True also returns the Stats."""
        scalar = np.ndim(seq) == 0 and np.ndim(begin) == 0 and np.ndim(end) == 0
        seq, begin, end = np.broadcast_arrays(_u64(seq).reshape(-1), _u64(begin).reshape(-1), _u64(end).reshape(-1))
        seq, begin, end = _u64(seq), _u64(begin), _u64(end)
        count = seq.size
        offsets = np.zeros(count + 1, dtype=np.uint64)
        need = int((end.astype(np.int64) - begin.astype(np.int64)).clip(min=0).sum()) if count else 0
        out = np.zeros(max(need, 1), dtype=np.uint8)
        st = Stats()
        _check(lib().fmb_extract(self.h, _ptr(seq), _ptr(begin), _ptr(end), C.c_uint64(count), _ptr(out), C.c_uint64(need),
                                 _ptr(offsets), C.byref(st)))
        parts = [out[offsets[i]:offsets[i + 1]] for i in range(count)]
        res = parts[0] if scalar else parts
        return (res, st) if with_stats else res

    def reconstruct_text(self):
        """reconstructText (utils.h:672): the text s0 0 s1 0 ... 0 the index was built from, n bytes"""
        out = np.zeros(self.info.n, dtype=np.uint8)
        _check(lib().fmb_index_reconstruct_text(self.h, _ptr(out), C.c_uint64(out.size)))
        return out

    def search_and_locate(self, symbols, offsets, scheme=None, partition=None, edit=False, capacity=None,
                          out=None, packed=None):
        """One-call host-to-host path (fmb_search_and_locate; with packed = pack_queries(symbols): fmb_search_and_locate_packed,
        symbols may then be None)."""
        symbols, offsets = (None if packed is not None else _u8(symbols)), _u64(offsets)
        nq = offsets.size - 1
        if scheme is None:
            ns, npart, pi, l, u, part = 0, 0, None, None, None, None
        else:
            pi, l, u = (np.ascontiguousarray(a, dtype=np.uint32) for a in scheme)
            part = _u32(partition)
            ns, npart = pi.shape
        if out is None:
            out = np.zeros(capacity if capacity is not None else max(nq, 1) * 4, dtype=LOC32_DTYPE)
        n_out = C.c_uint64(0)
        st = Stats()
        if packed is not None:
            words, exc_pos, exc_sym = packed
            words, exc_pos, exc_sym = np.ascontiguousarray(words, dtype=np.uint32), _u64(exc_pos), _u8(exc_sym)
            _check(lib().fmb_search_and_locate_packed(self.h, _ptr(words), _ptr(offsets), C.c_uint64(nq), _ptr(exc_pos), _ptr(exc_sym),
                                                      C.c_uint64(exc_pos.size), C.c_int(1 if edit else 0),
                                                      C.c_uint32(ns), C.c_uint32(npart), _ptr(pi), _ptr(l), _ptr(u), _ptr(part),
                                                      _ptr(out), C.c_uint64(out.size), C.byref(n_out), C.byref(st)))
            return out[: n_out.value], st
        _check(lib().fmb_search_and_locate(self.h, _ptr(symbols), _ptr(offsets), C.c_uint64(nq), C.c_int(1 if edit else 0),
                                           C.c_uint32(ns), C.c_uint32(npart), _ptr(pi), _ptr(l), _ptr(u), _ptr(part),
                                           _ptr(out), C.c_uint64(out.size), C.byref(n_out), C.byref(st)))
        return out[: n_out.value], st


def pack_queries(symbols, sigma=5, words=None):
    """2-bit packing of byte symbols (symbol - 1, 16 per little-endian word) + exception list (positions of symbols without 2-bit
    code: 0 and >= sigma), the input form of fmb_queries_upload_packed / fmb_search_and_locate_packed (host-side fmb_pack_symbols;
    `words`: optional destination, e.g. a view of pinned memory, of at least (n + 15) // 16 + 1 words)"""
    s = _u8(symbols)
    L = lib()
    L.fmb_pack_symbols.restype = C.c_uint64
    if words is None:
        words = np.zeros((s.size + 15) // 16 + 1, dtype=np.uint32)
    cap = 1024
    while True:
        exc_pos, exc_sym = np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.uint8)
        n = L.fmb_pack_symbols(_ptr(s), C.c_uint64(0), C.c_uint64(s.size), C.c_uint32(sigma), _ptr(words), _ptr(exc_pos), _ptr(exc_sym), C.c_uint64(cap))
        if n <= cap:
            return words, exc_pos[:n].copy(), exc_sym[:n].copy()
        cap = int(n)


def search_and_locate_multi(replicas, symbols, offsets, scheme=None, partition=None, edit=False, shard_capacity=None, out=None):
    """fmb_search_and_locate_multi: one call, the queries sharded contiguously over the replicas; returns (list of row arrays, stats)"""
    symbols, offsets = _u8(symbols), _u64(offsets)
    nq = offsets.size - 1
    G = len(replicas)
    if scheme is None:
        ns, npart, pi, l, u, part = 0, 0, None, None, None, None
    else:
        pi, l, u = (np.ascontiguousarray(a, dtype=np.uint32) for a in scheme)
        part = _u32(partition)
        ns, npart = pi.shape
    if shard_capacity is None:
        shard_capacity = (out.size // G) if out is not None else max((nq + G - 1) // G, 1) * 4
    if out is None:
        out = np.zeros(shard_capacity * G, dtype=LOC32_DTYPE)
    handles = (C.c_void_p * G)(*[r.h for r in replicas])
    n_out = (C.c_uint64 * G)()
    st = Stats()
    _check(lib().fmb_search_and_locate_multi(handles, C.c_uint32(G), _ptr(symbols), _ptr(offsets), C.c_uint64(nq), C.c_int(1 if edit else 0),
                                             C.c_uint32(ns), C.c_uint32(npart), _ptr(pi), _ptr(l), _ptr(u), _ptr(part),
                                             _ptr(out), C.c_uint64(shard_capacity), n_out, C.byref(st)))
    return [out[g * shard_capacity: g * shard_capacity + n_out[g]] for g in range(G)], st


def search_and_locate_parts(parts, seq_base, symbols, offsets, scheme=None, partition=None, edit=False, part_capacity=None):
    """fmb_search_and_locate_parts: a collection split into several indices over disjoint sequences; the whole batch is searched in every
    part, rows carry the sequence numbers of the whole collection; returns (list of row arrays, one per part, stats)"""
    symbols, offsets = _u8(symbols), _u64(offsets)
    nq = offsets.size - 1
    P = len(parts)
    if scheme is None:
        ns, npart, pi, l, u, part = 0, 0, None, None, None, None
    else:
        pi, l, u = (np.ascontiguousarray(a, dtype=np.uint32) for a in scheme)
        part = _u32(partition)
        ns, npart = pi.shape
    if part_capacity is None:
        part_capacity = max(nq, 1) * 4
    out = np.zeros(part_capacity * P, dtype=LOC32_DTYPE)
    handles = (C.c_void_p * P)(*[r.h for r in parts])
    bases = _u64(seq_base)
    n_out = (C.c_uint64 * P)()
    st = Stats()
    _check(lib().fmb_search_and_locate_parts(handles, C.c_uint32(P), _ptr(bases), _ptr(symbols), _ptr(offsets), C.c_uint64(nq), C.c_int(1 if edit else 0),
                                             C.c_uint32(ns), C.c_uint32(npart), _ptr(pi), _ptr(l), _ptr(u), _ptr(part),
                                             _ptr(out), C.c_uint64(part_capacity), n_out, C.byref(st)))
    return [out[g * part_capacity: g * part_capacity + n_out[g]] for g in range(P)], st


class Queries:
    def __init__(self, index, symbols, offsets, complement=None, packed=None):
        offsets = _u64(offsets)
        self.h = C.c_void_p()
        if packed is not None:
            words, exc_pos, exc_sym = packed
            words, exc_pos, exc_sym = np.ascontiguousarray(words, dtype=np.uint32), _u64(exc_pos), _u8(exc_sym)
            _check(lib().fmb_queries_upload_packed(C.byref(self.h), index.h, _ptr(words), _ptr(offsets), C.c_uint64(offsets.size - 1),
                                                   _ptr(exc_pos), _ptr(exc_sym), C.c_uint64(exc_pos.size)))
            return
        symbols = _u8(symbols)
        if complement is None:
            _check(lib().fmb_queries_upload(C.byref(self.h), index.h, _ptr(symbols), _ptr(offsets), C.c_uint64(offsets.size - 1)))
        else:
            comp = _u8(complement)
            _check(lib().fmb_queries_upload_revcomp(C.byref(self.h), index.h, _ptr(symbols), _ptr(offsets), C.c_uint64(offsets.size - 1), _ptr(comp)))

    def __len__(self):
        return lib().fmb_queries_count(self.h)

    def close(self):
        if self.h:
            lib().fmb_queries_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Results:
    def __init__(self, handle):
        self.h = handle

    def __len__(self):
        return lib().fmb_results_count(self.h)

    @property
    def kind(self):
        return lib().fmb_results_kind(self.h)

    @property
    def stats(self):
        s = Stats()
        _check(lib().fmb_results_get_stats(self.h, C.byref(s)))
        return s

    def hits(self):
        out = np.zeros(len(self), dtype=HIT_DTYPE)
        _check(lib().fmb_results_fetch_hits(self.h, _ptr(out), C.c_uint64(out.size)))
        return out

    def locs(self):
        out = np.zeros(len(self), dtype=LOC_DTYPE)
        _check(lib().fmb_results_fetch_locs(self.h, _ptr(out), C.c_uint64(out.size)))
        return out

    def locs32(self):
        out = np.zeros(len(self), dtype=LOC32_DTYPE)
        _check(lib().fmb_results_fetch_locs32(self.h, _ptr(out), C.c_uint64(out.size)))
        return out

    def smems(self):
        """SMEM records (qidx, begin, end, lb, len) of fmb_search_smems"""
        out = np.zeros(len(self), dtype=SMEM_DTYPE)
        _check(lib().fmb_results_fetch_smems(self.h, _ptr(out), C.c_uint64(out.size)))
        return out

    def smem_locs(self):
        """located SMEM rows (qidx, begin, end, seq, pos) of fmb_locate_smems"""
        out = np.zeros(len(self), dtype=SMEM_LOC_DTYPE)
        _check(lib().fmb_results_fetch_smem_locs(self.h, _ptr(out), C.c_uint64(out.size)))
        return out

    def close(self):
        if self.h:
            lib().fmb_results_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- raw-pointer helpers (bench / synthetic workloads) ---------------------------------------------------
class PinnedArray:
    """numpy view over page-locked host memory from fmb_host_alloc_pinned (fast H2D / D2H)"""

    def __init__(self, count, dtype):
        self.dtype = np.dtype(dtype)
        self.nbytes = int(count) * self.dtype.itemsize
        self.ptr = lib().fmb_host_alloc_pinned(C.c_uint64(max(self.nbytes, 1)))
        if not self.ptr:
            raise FmbError(-4, lib().fmb_last_error().decode())
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(count))

    def free(self):
        if self.ptr:
            self.array = None
            lib().fmb_host_free_pinned(C.c_void_p(self.ptr))
            self.ptr = None


def synth_text_device(device, sigma, n, seed):
    p = C.c_void_p()
    _check(lib().fmb_synth_text_device(C.c_int(device), C.c_uint32(sigma), C.c_uint64(n), C.c_uint64(seed), C.byref(p)))
    return p.value


def synth_reads_device(device, d_text, n, nq, length, seed):
    p = C.c_void_p()
    _check(lib().fmb_synth_reads_device(C.c_int(device), C.c_void_p(d_text), C.c_uint64(n), C.c_uint64(nq), C.c_uint32(length),
                                        C.c_uint64(seed), C.byref(p)))
    return p.value


def synth_reads_err_device(device, d_text, n, nq, length, seed, sigma, max_errors, edit):
    p = C.c_void_p()
    _check(lib().fmb_synth_reads_err_device(C.c_int(device), C.c_void_p(d_text), C.c_uint64(n), C.c_uint64(nq), C.c_uint32(length),
                                            C.c_uint64(seed), C.c_uint32(sigma), C.c_uint32(max_errors), C.c_int(1 if edit else 0), C.byref(p)))
    return p.value


def synth_repeat_text_device(device, sigma, n, seed, unit_len, copies, sub_per_mille):
    p = C.c_void_p()
    _check(lib().fmb_synth_repeat_text_device(C.c_int(device), C.c_uint32(sigma), C.c_uint64(n), C.c_uint64(seed), C.c_uint32(unit_len),
                                              C.c_uint32(copies), C.c_uint32(sub_per_mille), C.byref(p)))
    return p.value


def synth_unit_reads_device(device, sigma, nq, length, seed, unit_len):
    p = C.c_void_p()
    _check(lib().fmb_synth_unit_reads_device(C.c_int(device), C.c_uint32(sigma), C.c_uint64(nq), C.c_uint32(length), C.c_uint64(seed),
                                             C.c_uint32(unit_len), C.byref(p)))
    return p.value


def device_free(device, ptr):
    _check(lib().fmb_device_free(C.c_int(device), C.c_void_p(ptr)))


def copy_to_host(device, host_array, d_ptr, nbytes):
    _check(lib().fmb_copy_to_host(C.c_int(device), _ptr(host_array), C.c_void_p(d_ptr), C.c_uint64(nbytes)))


def kernel_launch_count():
    return int(lib().fmb_kernel_launch_count())


def measure_gather(index, table, requests=1 << 28):
    """independent random gathers over one of the index's tables: (requests per second, table bytes, bytes per request)"""
    rps, tb, rb = C.c_double(0), C.c_uint64(0), C.c_uint32(0)
    _check(lib().fmb_measure_gather(index.h, C.c_int(table), C.c_uint64(requests), C.byref(rps), C.byref(tb), C.byref(rb)))
    return rps.value, tb.value, rb.value


def set_image_budget(nbytes):
    """HBM budget of the index images created after this call (0 = no limit)"""
    _check(lib().fmb_set_image_budget(C.c_uint64(int(nbytes))))


def index_set_stream(index, stream_ptr):
    _check(lib().fmb_index_set_stream(index.h, C.c_void_p(stream_ptr)))
