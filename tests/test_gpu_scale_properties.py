"""Size-independent properties at a scale the oracle would take minutes for (64 Mbp index built on the GPU, 10^6 reads): the
accelerating tables (k-mer tables, pair table, LF^16 jumps in both directions, locate shortcut) are all exercised at realistic
interval widths.  Reads are copied from known text offsets, so the expected answers follow from the construction."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N_TEXT = 64_000_000
NQ = 1_000_000
L = 150


@pytest.fixture(scope="module")
def big(gpu):
    from fmb200 import capi
    d_text = capi.synth_text_device(0, 5, N_TEXT, 11)
    index = gpu.Index.build_from_device_text(5, d_text, N_TEXT, sampling_rate=16, bidirectional=True, device=0)
    yield gpu, capi, index, d_text
    capi.device_free(0, d_text)


def _reads(capi, d_text, kind, k=0, edit=False, length=L, nq=NQ):
    if kind == "exact":
        d = capi.synth_reads_device(0, d_text, N_TEXT, nq, length, 12)
    else:
        d = capi.synth_reads_err_device(0, d_text, N_TEXT, nq, length, 12, 5, k, edit)
    sym = np.zeros(nq * length, dtype=np.uint8)
    capi.copy_to_host(0, sym, d, nq * length)
    capi.device_free(0, d)
    return sym, np.arange(nq + 1, dtype=np.uint64) * np.uint64(length)


@pytest.fixture(scope="module")
def big_oracle(big):
    """the oracle on the device index's own BWT and samples (its checkpoints take ~5 MB per direction at this size)"""
    from oracle.pyoracle import Oracle
    gpu, capi, index, _ = big
    return Oracle.from_bwt(5, *index.export())


SAMPLE = 2000


def _sample_parity(index, o, search, sym, off, res, length, locate=True):
    """the device's hits (and located rows) of a fixed sample of SAMPLE reads of the whole batch == the oracle's for those reads alone
    (search(symbols, offsets): the oracle's hits)"""
    from helpers import hits_equal, locs_equal
    nq = off.size - 1
    size = min(SAMPLE, nq)
    sample = np.sort(np.random.default_rng(2024).choice(nq, size, replace=False)).astype(np.uint64)
    renum = np.full(nq, -1, dtype=np.int64)
    renum[sample] = np.arange(size)
    ssym = sym.reshape(nq, length)[sample].reshape(-1)
    soff = np.arange(size + 1, dtype=np.uint64) * np.uint64(length)
    hits = res.hits()
    got = hits[renum[hits["qidx"].astype(np.int64)] >= 0]
    got["qidx"] = renum[got["qidx"].astype(np.int64)]
    exp = search(ssym, soff)
    assert len(exp) >= size // 2
    assert hits_equal(got, exp)
    if locate:
        locs = index.locate(res).locs()
        gl = locs[renum[locs["qidx"].astype(np.int64)] >= 0]
        gl["qidx"] = renum[gl["qidx"].astype(np.int64)]
        assert locs_equal(gl, o.locate(exp))


def _source_offsets():
    from fmb200 import synth
    i = np.arange(NQ, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = synth.splitmix64(i * np.uint64(0x632BE59BD9B4E019) + np.uint64(12))
    return (z % np.uint64(N_TEXT - L)).astype(np.uint64)


def _has_deletion(k):
    """which reads of synth_reads_err_kernel (seed 12, edit mode) contain a planted deletion: such a read ends in a random symbol,
    so it may need one more error than was planted and is not guaranteed to be found"""
    from fmb200 import synth
    q = np.arange(NQ, dtype=np.uint64)
    with np.errstate(over="ignore"):
        h = synth.splitmix64(q * np.uint64(0x9E3779B97F4A7C15) + np.uint64(12 * 31 + 7))
        ne = h % np.uint64(k + 1)
        has = np.zeros(NQ, dtype=bool)
        for i in range(k):
            h = synth.splitmix64(h + np.uint64(i + 1))
            has |= (ne > i) & (h % np.uint64(3) == 2)
    return has


def test_tables_present(big):
    gpu, capi, index, _ = big
    assert index.info.tables & 0x7F == 0x7F          # pair, kmer, jump, jump_rev, locblock, locrow, bikmer
    assert index.info.tables & 0x180 == 0x180        # LF^4 tables, merged LF^16 / LF^32 entries in direction 0


def test_narrow_jump_table_gives_the_same_answers(gpu):
    """FMB_NO_JUMP32 (read when an index is built) keeps the 8-byte LF^16 entries: the exact-search and scheme parity tests again
    in a fresh process"""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, FMB_NO_JUMP32="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_string_and_exact.py"),
                        os.path.join(root, "tests", "test_gpu_scheme_and_build.py"), "-q", "-x"], env=env, capture_output=True, text=True, timeout=900, cwd=root)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_exact_reads_are_found_where_they_came_from(big):
    gpu, capi, index, d_text = big
    sym, off = _reads(capi, d_text, "exact")
    q = index.upload(sym, off)
    res = index.search_exact(q)
    hits = res.hits()
    assert len(hits) == NQ and np.array_equal(hits["qidx"], np.arange(NQ, dtype=np.uint64))      # every read occurs, one cursor each
    assert np.all(hits["steps"] == L) and np.all(hits["len"] >= 1)
    src = _source_offsets()
    locs = index.locate(res).locs()
    found = np.zeros(NQ, dtype=bool)
    found[locs["qidx"][locs["pos"] == src[locs["qidx"]]]] = True
    assert found.all()                                                                              # the source offset is among the located rows
    # the three exact kernels / two locate kernels agree with each other
    index.set_exact_mode(1)
    h1 = index.search_exact(q).hits()
    index.set_exact_mode(0)
    assert np.array_equal(h1, hits)
    index.set_locate_mode(1)
    walk = index.locate(res).locs()
    index.set_locate_mode(0)
    assert np.array_equal(np.sort(walk, order=["qidx", "seq", "pos", "e"]), np.sort(locs, order=["qidx", "seq", "pos", "e"]))
    # one-call host path = the same rows
    rows, _ = index.search_and_locate(sym, off, capacity=NQ + 1000)
    assert np.array_equal(np.sort(rows, order=["qidx", "seq", "pos", "e"])["pos"], np.sort(locs, order=["qidx", "seq", "pos", "e"])["pos"].astype(np.uint32))


@pytest.mark.parametrize("k,edit", [(1, False), (2, False), (1, True), (2, True)])
def test_reads_with_planted_errors_are_found(big, k, edit):
    """a read with e <= k planted edits must be reported with some error count <= k at (or, for edit distance, next to) its source
    offset; Hamming hits additionally have steps == L and e equal to the number of differing symbols"""
    from fmb200 import schemes
    gpu, capi, index, d_text = big
    sym, off = _reads(capi, d_text, "err", k, edit)
    sch = schemes.optimum(0, k)
    part = schemes.uniform_partition(sch[0].shape[1], L)
    res = index.search_scheme(index.upload(sym, off), sch, part, edit)
    hits = res.hits()
    assert np.all(hits["e"] <= k) and np.all(hits["len"] >= 1)
    if not edit:
        assert np.all(hits["steps"] == L)
    else:
        assert np.all(np.abs(hits["steps"].astype(np.int64) - L) <= k)
    must = ~_has_deletion(k) if edit else np.ones(NQ, dtype=bool)
    src = _source_offsets()
    locs = index.locate(res).locs()
    near = np.abs(locs["pos"].astype(np.int64) - src[locs["qidx"]].astype(np.int64)) <= (k if edit else 0)
    found = np.zeros(NQ, dtype=bool)
    found[locs["qidx"][near]] = True
    assert found[must].all()                                                                        # found at (next to) the source offset
    assert must.mean() > 0.6
    # the jump / k-mer accelerated kernel and the plain frontier kernel report the same multiset
    st = res.stats
    assert 0 < st.line_requests < st.occ_lookups


@pytest.mark.parametrize("k,edit", [(1, False), (2, False), (1, True), (2, True)])
def test_sample_of_the_batch_matches_oracle(big, big_oracle, k, edit):
    """the whole 10^6-read batch on the device; the hits and located rows of a fixed sample of 2000 reads equal the oracle's"""
    from fmb200 import schemes
    gpu, capi, index, d_text = big
    sym, off = _reads(capi, d_text, "err", k, edit)
    sch = schemes.optimum(0, k)
    part = schemes.uniform_partition(sch[0].shape[1], L)
    res = index.search_scheme(index.upload(sym, off), sch, part, edit)
    _sample_parity(index, big_oracle, lambda s, f: big_oracle.search_ng26(s, f, sch, part, edit), sym, off, res, L)


def _bikmer_k(n):
    """k of the bidirectional k-mer table of a DNA index of n rows (csrc/fmb_lib.cu build_bikmer): the largest k <= 14 with 8 * 4^k <= n"""
    k = 0
    while k < 14 and 8 << (2 * (k + 1)) <= n:
        k += 1
    return k


@pytest.mark.parametrize("length", [24, 40])
@pytest.mark.parametrize("edit", [False, True])
def test_short_reads_skip_the_bidirectional_kmer_table(big, big_oracle, length, edit):
    """k = 2 on 24- and 40-symbol reads: the error-free first parts (6 and 10 symbols) are shorter than the bidirectional k-mer
    table's k, so the roots start at the full interval and the wide-interval phase runs on the index.  (Such reads have hundreds of
    single-row paths per root: batches much larger than these exceed the frontier lists, which the search reports as FMB_EOVERFLOW.)"""
    from fmb200 import schemes
    gpu, capi, index, d_text = big
    sch = schemes.optimum(0, 2)
    part = schemes.uniform_partition(sch[0].shape[1], length)
    bk = _bikmer_k(index.info.n)
    assert bk == 11 and max(part) < bk
    sym, off = _reads(capi, d_text, "err", 2, edit, length, {24: 250, 40: 1500}[length])
    res = index.search_scheme(index.upload(sym, off), sch, part, edit)
    _sample_parity(index, big_oracle, lambda s, f: big_oracle.search_ng26(s, f, sch, part, edit), sym, off, res, length)


@pytest.mark.parametrize("length", [8, 10, 11, 12, 13, 16])
def test_exact_reads_around_the_kmer_table_k(big, big_oracle, length):
    """exact search of reads as long as the exact k-mer table's k (11 here) and around it; located rows for the reads of 12 symbols and
    more (the shorter ones have intervals of hundreds of rows)"""
    gpu, capi, index, d_text = big
    sym, off = _reads(capi, d_text, "exact", length=length, nq=200_000)
    res = index.search_exact(index.upload(sym, off))
    _sample_parity(index, big_oracle, big_oracle.search_exact, sym, off, res, length, locate=length >= 12)


@pytest.mark.parametrize("k,edit", [(1, False), (2, True)])
def test_hit_limit_properties_at_scale(big, k, edit):
    """search_n at 10^6 reads: the limited lists nest (the list for n is a prefix, per query, of the list for a larger n, the last
    cursor possibly clipped), every query with a hit keeps one, no query exceeds n rows, and the unlimited search reports the
    same multiset as the ordered one with n = infinity"""
    from fmb200 import schemes
    gpu, capi, index, d_text = big
    sym, off = _reads(capi, d_text, "err", k, edit)
    q = index.upload(sym, off)
    sch = schemes.optimum(0, k)
    part = schemes.uniform_partition(sch[0].shape[1], L)
    full = index.search_scheme(q, sch, part, edit).hits()
    order = ["qidx", "e", "lb", "len", "steps", "lb_rev"]
    big_n = index.search_scheme(q, sch, part, edit, n=10**12).hits()
    assert np.array_equal(np.sort(full, order=order), np.sort(big_n, order=order))
    assert np.all(np.diff(big_n["qidx"].astype(np.int64)) >= 0)                   # grouped by ascending qidx
    prev = big_n
    for n in (3, 1):
        lim = index.search_scheme(q, sch, part, edit, n=n).hits()
        rows = np.bincount(lim["qidx"].astype(np.int64), weights=lim["len"].astype(np.float64), minlength=NQ)
        rows_full = np.bincount(full["qidx"].astype(np.int64), weights=full["len"].astype(np.float64), minlength=NQ)
        assert np.array_equal(rows, np.minimum(rows_full, n))                      # exactly min(n, all rows) rows per query
        # prefix property: the j-th hit of a query in `lim` is the j-th hit of that query in `prev` (len possibly clipped)
        def rank_in_query(h):
            first = np.searchsorted(h["qidx"], h["qidx"], side="left")
            return np.arange(len(h)) - first
        pos_prev = np.searchsorted(prev["qidx"], lim["qidx"], side="left") + rank_in_query(lim)
        same = prev[pos_prev]
        for f in ("qidx", "lb", "lb_rev", "steps", "e"):
            assert np.array_equal(lim[f], same[f]), (n, f)
        assert np.all(lim["len"] <= same["len"])
        prev = lim


def test_locate_refuses_more_than_2_32_rows(big):
    """300 one-symbol queries cover ~4.8 G rows of the 64 Mbp index: locate must fail loudly, not wrap around"""
    gpu, capi, index, _ = big
    sym = np.tile(np.array([1, 2, 3, 4], dtype=np.uint8), 75)
    off = np.arange(301, dtype=np.uint64)
    res = index.search_exact(index.upload(sym, off))
    hits = res.hits()
    assert len(hits) == 300 and int(hits["len"].sum()) > 2 ** 32
    with pytest.raises(gpu.FmbError) as ei:
        index.locate(res)
    assert ei.value.code == -6 and "split the batch" in str(ei.value)
