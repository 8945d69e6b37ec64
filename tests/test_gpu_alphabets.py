"""Every kind of alphabet the library accepts (sigma = 2 .. 32) against the oracle.

Which device code an index runs depends on sigma.  sigma <= 5 takes the DNA layout: 2-bit codes, so sigma = 3 and 4 leave codes
unused and sigma = 2 is a text of one symbol, whose intervals stay wide.  Larger alphabets take the generic layout, whose 64-row blocks
hold ceil(log2 sigma) bit planes and sigma - 1 prefix counts in 64, 96, 128, 160 or 192 bytes; odd plane counts leave count words in
the last 16-byte plane load.  The k-error kernels (child mask up to sigma = 28), the keys of the hit-limited search, the byte-symbol
jump tables and the bidirectional k-mer table depend on sigma as well.  Each sigma below stands for one such case; every GPU test
builds its index pair once per sigma (the module fixture `alpha`)."""
from types import SimpleNamespace

import numpy as np
import pytest

from helpers import Oracle, hits_equal, locs_equal, make_index_pair, strip_lb_rev
from test_gpu_extract import check_index

SIGMAS = [2, 3, 4, 5, 6, 9, 12, 16, 17, 23, 24, 28, 31, 32]
DNA_SIGMAS = [2, 3, 4]                                   # DNA layout with unused 2-bit codes
SCHEME_SIGMAS = [s for s in SIGMAS if s <= 28]           # k-error searches
LENGTHS = [20000, 3000, 500, 64, 63, 1]
RATE = 4
READ_LENGTHS = [1, 2, 3, 4, 7, 8, 13, 14, 15, 16, 17, 31, 32, 33, 64, 100]
FMB_EUNSUPPORTED = -5
FMB_TABLE_PAIR = 1

# bytes per 64-row block of the occurrence table: 32 on the DNA layout, else roundup32(8 * planes + 4 * (sigma - 1))
OCC_BLOCK_BYTES = {2: 32, 3: 32, 4: 32, 5: 32, 6: 64, 9: 64, 12: 96, 16: 96, 17: 128, 23: 128, 24: 160, 28: 160, 31: 160, 32: 192}
# info.tables of each fixture's index (FMB_TABLE_* bits, see test_gpu_image_tables.py), bidirectional and unidirectional, as a B200
# build reports them: every table on the DNA layout; LF^4, locate shortcut and bidirectional k-mer table on the generic layout
TABLES = {s: 511 if s <= 5 else 224 for s in SIGMAS}
TABLES_UNIDIRECTIONAL = {s: 439 if s <= 5 else 160 for s in SIGMAS}


def on_gpu(sigmas):
    """the GPU cases of a test: one per sigma, each on the index pair of the `alpha` fixture"""
    def deco(f):
        return pytest.mark.gpu(pytest.mark.parametrize("alpha", sigmas, indirect=True, ids=[f"sigma{s}" for s in sigmas])(f))
    return deco


@pytest.fixture(scope="module")
def alpha(request, gpu):
    from fmb200 import synth
    sigma = request.param
    text = synth.multi_text(LENGTHS, sigma, 40 + sigma)
    o, g = make_index_pair(gpu, text, sigma, RATE)
    # (extraction adds a table on first use: the tables are read before any test runs)
    return SimpleNamespace(sigma=sigma, text=text, o=o, g=g, tables=g.info.tables)


def _sequences(text):
    ends = np.flatnonzero(text == 0)
    starts = np.concatenate([[0], ends[:-1] + 1])
    return [text[b:e] for b, e in zip(starts, ends)]


def _oracle_exact(o, reads, sigma, counters=None):
    """the oracle's exact-search hits of `reads` with the batch's query numbers; a read holding a symbol outside the alphabet (>= sigma)
    occurs nowhere and has no hit (the oracle itself only takes symbols < sigma)"""
    from fmb200 import synth
    valid = np.array([i for i, r in enumerate(reads) if not np.any(np.asarray(r) >= sigma)], dtype=np.int64)
    sym, off = synth.flatten([reads[i] for i in valid])
    hits = o.search_exact(sym, off, counters)
    hits["qidx"] = valid[hits["qidx"].astype(np.int64)].astype(np.uint64)
    return hits


def _plant(reads, sigma, n_err, edit, seed):
    """synth.plant_errors, except at sigma = 2: one letter leaves no substitution, so edit distance plants insertions and deletions only
    and Hamming distance plants nothing"""
    from fmb200 import synth
    if sigma > 2:
        return synth.plant_errors(reads, sigma, n_err, edit, seed)
    out = reads.copy()
    if not edit:
        return out
    rng = np.random.default_rng(seed)
    L = out.shape[1]
    for q in range(out.shape[0]):
        r = list(out[q])
        for _ in range(n_err):
            p = int(rng.integers(1, L - 1))
            if rng.integers(0, 2):
                r.insert(p, 1)
                r.pop()
            else:
                r.pop(p)
                r.append(1)
        out[q] = r
    return out


def _error_reads(alpha, nq, L, seed, edit):
    """reads from the first sequence: a third exact, a third with one error, a third with two.  sigma = 2 matches every position of
    the one-letter text, so a few reads keep the located rows below ~2 M"""
    from fmb200 import synth
    nq = nq if alpha.sigma > 2 else 6
    reads, _ = synth.reads_from_text(alpha.text[:LENGTHS[0] + 1], nq, L, seed)
    reads[nq // 3: 2 * nq // 3] = _plant(reads[nq // 3: 2 * nq // 3], alpha.sigma, 1, edit, seed + 1)
    reads[2 * nq // 3:] = _plant(reads[2 * nq // 3:], alpha.sigma, 2, edit, seed + 2)
    return synth.flatten(reads)


# ---- 1. layout, tables, GPU construction ----------------------------------------------------------------------------------------

@on_gpu(SIGMAS)
def test_layout_and_tables(alpha):
    sigma, text, o, g = alpha.sigma, alpha.text, alpha.o, alpha.g
    i = g.info
    assert i.sigma == sigma and i.n == text.size and i.bidirectional == 1 and i.n_delims == len(LENGTHS)
    assert i.occ_block_bytes == OCC_BLOCK_BYTES[sigma] and i.occ_block_rows == 64
    assert alpha.tables == TABLES[sigma]
    assert np.array_equal(g.C, o.C)
    bwt, rev, bm, sq, sp = g.export()
    obm, osq, osp = o.samples
    assert np.array_equal(bwt, o.bwt) and np.array_equal(rev, o.bwt_rev)
    assert np.array_equal(bm, obm) and np.array_equal(sq, osq) and np.array_equal(sp, osp)
    for dir in (0, 1):
        blocks, stride = g.export_blocks(dir)
        assert stride == OCC_BLOCK_BYTES[sigma] and blocks.size >= (text.size // 64 + 1) * stride


@on_gpu(SIGMAS)
@pytest.mark.parametrize("bidirectional", [True, False], ids=["bi", "uni"])
def test_gpu_build(gpu, alpha, bidirectional):
    """suffix sort, BWT, reverse BWT and text-space sampling on the GPU equal the oracle's; sigma = 2 holds a run of 20000 equal
    symbols, the deepest case of the prefix doubling"""
    sigma, text = alpha.sigma, alpha.text
    o = alpha.o if bidirectional else Oracle.build(text, sigma, RATE, False)
    g = gpu.Index.build(sigma, text, sampling_rate=RATE, bidirectional=bidirectional)
    bwt, rev, bm, sq, sp = g.export()
    assert np.array_equal(bwt, o.bwt)
    if bidirectional:
        assert np.array_equal(rev, o.bwt_rev)
    assert g.info.tables == (TABLES if bidirectional else TABLES_UNIDIRECTIONAL)[sigma]
    obm, osq, osp = o.samples
    assert np.array_equal(bm, obm) and np.array_equal(sq, osq) and np.array_equal(sp, osp)
    assert np.array_equal(g.C, o.C)
    assert g.info.occ_block_bytes == OCC_BLOCK_BYTES[sigma]
    assert gpu.Index.from_bwt(sigma, bwt, rev, bm, sq, sp).info.tables == g.info.tables


# ---- 2. String_c and cursors ----------------------------------------------------------------------------------------------------

def _probe_rows(n):
    """rows 0..n (rank takes n): the first and last 512, and +-2 around every multiple of 64 (block edges)"""
    edges = (np.arange(0, n + 1, 64)[:, None] + np.arange(-2, 3)[None, :]).ravel()
    rows = np.unique(np.concatenate([np.arange(512), np.arange(n - 511, n + 1), edges]))
    return rows[(rows >= 0) & (rows <= n)].astype(np.uint64)


@on_gpu(SIGMAS)
@pytest.mark.parametrize("dir", [0, 1])
def test_string_ops(alpha, dir):
    sigma, o, g = alpha.sigma, alpha.o, alpha.g
    n = o.n
    rows = _probe_rows(n)
    srows = rows[rows < n]
    assert np.array_equal(g.symbol(srows, dir), np.array([o.symbol(i, dir) for i in srows], dtype=np.uint8))
    # rank of every symbol, prefix_rank of every symbol and of sigma itself
    for fn, ofn, top in ((g.rank, o.rank, sigma), (g.prefix_rank, o.prefix_rank, sigma + 1)):
        idx = np.repeat(rows, top)
        symb = np.tile(np.arange(top, dtype=np.uint8), rows.size)
        exp = np.array([ofn(i, s, dir) for i, s in zip(idx, symb)], dtype=np.uint64)
        assert np.array_equal(fn(idx, symb, dir), exp), ofn.__name__
    rng = np.random.default_rng(10 * sigma + dir)
    idx = rng.integers(0, n + 1, size=5000).astype(np.uint64)
    symb = rng.integers(0, sigma, size=5000).astype(np.uint8)
    assert np.array_equal(g.rank(idx, symb, dir), np.array([o.rank(i, s, dir) for i, s in zip(idx, symb)], dtype=np.uint64))
    symb = rng.integers(0, sigma + 1, size=5000).astype(np.uint8)
    assert np.array_equal(g.prefix_rank(idx, symb, dir), np.array([o.prefix_rank(i, s, dir) for i, s in zip(idx, symb)], dtype=np.uint64))
    rs, prs = g.all_ranks(rows, dir)
    for k, i in enumerate(rows):
        ors, oprs = o.all_ranks_and_prefix_ranks(int(i), dir)
        assert np.array_equal(rs[k], ors) and np.array_equal(prs[k], oprs), int(i)
    # every row and every symbol against plain counts over the BWT
    bwt = o.bwt if dir == 0 else o.bwt_rev
    counts = np.zeros((n + 1, sigma), dtype=np.uint64)
    counts[1:] = np.cumsum(bwt[:, None] == np.arange(sigma, dtype=np.uint8)[None, :], axis=0)
    less = np.zeros((n + 1, sigma + 1), dtype=np.uint64)
    less[:, 1:] = np.cumsum(counts, axis=1)
    every = np.arange(n + 1, dtype=np.uint64)
    rs, prs = g.all_ranks(every, dir)
    assert np.array_equal(rs, counts) and np.array_equal(prs, less[:, :sigma])
    idx = np.repeat(every, sigma + 1)
    symb = np.tile(np.arange(sigma + 1, dtype=np.uint8), n + 1)
    assert np.array_equal(g.prefix_rank(idx, symb, dir), less.ravel())
    assert np.array_equal(g.symbol(every[:-1], dir), bwt)


@on_gpu(SIGMAS)
def test_cursor_extend(alpha):
    sigma, o, g = alpha.sigma, alpha.o, alpha.g
    rng = np.random.default_rng(sigma)
    # cursors reached by real searches: start from the root and extend randomly, keep the non-empty ones
    curs = [np.array([0, 0, o.n, 0], dtype=np.uint64)]
    for _ in range(400):
        c = curs[rng.integers(0, len(curs))]
        nc = o.extend(c, int(rng.integers(0, sigma)), bool(rng.integers(0, 2)))
        if nc[2] > 0:
            curs.append(nc)
    curs = np.array(curs, dtype=np.uint64)
    assert len(curs) > 100
    for right in (0, 1):
        for s in range(sigma):
            got = g.extend(curs, np.full(len(curs), s, dtype=np.uint8), right)
            exp = np.array([o.extend(c, s, right) for c in curs], dtype=np.uint64)
            assert np.array_equal(got, exp), (right, s)
        got = g.extend_all(curs, right)
        exp = np.array([o.extend_all(c, right) for c in curs], dtype=np.uint64)
        assert np.array_equal(got, exp), right


# ---- 3. exact search and locate -------------------------------------------------------------------------------------------------

def _exact_reads(text, sigma, seed):
    """reads copied from the text (they may straddle delimiters), random reads, reads holding symbol 0 and, below sigma = 5, reads
    holding a 2-bit code that is no symbol of the alphabet (sigma .. 4).  sigma = 2: every copied read matches most of the text, so
    fewer of them keep locate's rows near a million"""
    rng = np.random.default_rng(seed)
    per = 24 if sigma > 2 else 2
    reads = []
    for L in READ_LENGTHS:
        for _ in range(per):
            p = int(rng.integers(0, text.size - L))
            reads.append(text[p:p + L].copy())
        for _ in range(max(per // 4, 1)):
            reads.append(rng.integers(1, sigma, size=L).astype(np.uint8))
            reads.append(rng.integers(0, sigma, size=L).astype(np.uint8))
        if sigma < 5:
            for _ in range(max(per // 4, 1)):
                p = int(rng.integers(0, LENGTHS[0] - L))
                r = text[p:p + L].copy()
                r[rng.integers(0, L)] = rng.integers(sigma, 5)
                reads.append(r)
    return reads


@on_gpu(SIGMAS)
def test_exact_search_and_locate(alpha):
    from fmb200 import synth
    from oracle.pyoracle import Counters
    sigma, text, o, g = alpha.sigma, alpha.text, alpha.o, alpha.g
    reads = _exact_reads(text, sigma, 3 + sigma)
    sym, off = synth.flatten(reads)
    q = g.upload(sym, off)
    exp = _oracle_exact(o, reads, sigma)
    assert len(exp) > 0
    modes = (0, 1, 2) if alpha.tables & FMB_TABLE_PAIR else (0, 1)      # 2: the two-symbol kernel of the DNA layout
    try:
        for mode in modes:
            g.set_exact_mode(mode)
            res = g.search_exact(q)
            got = res.hits()
            assert hits_equal(got, exp), mode
            assert np.all(np.diff(got["qidx"].astype(np.int64)) > 0)
    finally:
        g.set_exact_mode(0)
    res = g.search_exact(q)
    exp_locs = o.locate(exp)
    try:
        for mode in (0, 1):                                             # 1: walk LF steps, no shortcut table
            g.set_locate_mode(mode)
            loc = g.locate(res)
            locs = loc.locs()
            assert locs_equal(locs, exp_locs), mode
            assert np.array_equal(loc.locs32()["pos"].astype(np.uint64), locs["pos"])
            assert np.array_equal(loc.locs32()["seq"].astype(np.uint64), locs["seq"])
            ctr = Counters()
            o.locate(exp, ctr)
            assert loc.stats.lf_steps == ctr.lf_steps, mode
    finally:
        g.set_locate_mode(0)
    # the work counters of the one-symbol kernel (reads the oracle can search: symbols < sigma)
    valid = [r for r in reads if not np.any(r >= sigma)]
    vsym, voff = synth.flatten(valid)
    ctr = Counters()
    vexp = o.search_exact(vsym, voff, ctr)
    try:
        g.set_exact_mode(1)
        st = g.search_exact(g.upload(vsym, voff)).stats
    finally:
        g.set_exact_mode(0)
    assert len(vexp) > 0 and st.extensions == ctr.extensions and st.occ_lookups == ctr.occ_lookups


@on_gpu(SIGMAS)
def test_locate_rows_and_samples(alpha):
    o, g = alpha.o, alpha.g
    rows = np.arange(o.n, dtype=np.uint64)
    seq, pos, steps = g.locate_rows(rows)
    exp = np.array([o.locate_row(int(r)) for r in rows], dtype=np.uint64).reshape(-1, 3)
    assert np.array_equal(seq.astype(np.uint64), exp[:, 0]) and np.array_equal(pos.astype(np.uint64), exp[:, 1])
    assert np.array_equal(steps, exp[:, 2])
    has, sseq, spos = g.sample_value(rows)
    osv = [o.single_locate_step(int(r)) for r in rows]
    assert np.array_equal(has.astype(bool), np.array([v is not None for v in osv]))
    on = np.flatnonzero(has)
    assert np.array_equal(sseq[on], np.array([osv[i][0] for i in on], dtype=np.uint32))
    assert np.array_equal(spos[on], np.array([osv[i][1] for i in on], dtype=np.uint32))


@on_gpu(DNA_SIGMAS)
def test_packed_queries_and_reverse_complement(alpha):
    """2-bit packed queries on a DNA-layout index with unused codes: packed for this sigma (symbols sigma .. 4 go to the exception
    list) and for sigma = 5 (they travel as 2-bit codes, and the device must flag them after unpacking); the one-call path; and the
    reverse-complement doubling with a sigma-entry complement table"""
    from fmb200 import capi, schemes, synth
    sigma, text, o, g = alpha.sigma, alpha.text, alpha.o, alpha.g
    rng = np.random.default_rng(sigma)
    L, nq = 24, (300 if sigma > 2 else 12)
    reads, _ = synth.reads_from_text(text[:LENGTHS[0] + 1], nq, L, 17)
    for i in range(0, nq, 7):
        reads[i, rng.integers(0, L)] = 0
    for i in range(3, nq, 5):
        reads[i, rng.integers(0, L)] = rng.integers(sigma, 5)
    sym, off = synth.flatten(reads)
    exp = _oracle_exact(o, list(reads), sigma)
    exp_locs = o.locate(exp)
    assert len(exp) > 0

    def as_locs(rows):
        out = np.zeros(len(rows), dtype=exp_locs.dtype)
        for f in ("qidx", "seq", "pos", "e"):
            out[f] = rows[f]
        return out

    own, five = capi.pack_queries(sym, sigma), capi.pack_queries(sym)
    assert five[1].size < own[1].size                   # symbols sigma .. 4 are no exceptions when packed for sigma = 5
    for packed in (own, five):
        assert hits_equal(g.search_exact(g.upload(None, off, packed=packed)).hits(), exp)
        locs, _ = g.search_and_locate(None, off, packed=packed, capacity=len(exp_locs) + 16)
        assert locs_equal(as_locs(locs), exp_locs)
    locs, _ = g.search_and_locate(sym, off, capacity=len(exp_locs) + 16)
    assert locs_equal(as_locs(locs), exp_locs)
    # a k = 1 search through the one-call path, reads with symbols of the alphabet only
    ok = ~np.any(reads >= sigma, axis=1)
    vsym, voff = synth.flatten(reads[ok])
    sch, part = schemes.optimum(0, 1), schemes.uniform_partition(2, L)
    sexp = o.locate(o.search_ng26(vsym, voff, sch, part, True))
    for packed in (None, capi.pack_queries(vsym, sigma), capi.pack_queries(vsym)):
        locs, _ = g.search_and_locate(vsym if packed is None else None, voff, scheme=sch, partition=part, edit=True,
                                      capacity=len(sexp) + 16, packed=packed)
        assert locs_equal(as_locs(locs), sexp)
    # reverse complement: 1 <-> sigma - 1, 2 <-> sigma - 2, ...
    comp = np.array([0] + [sigma - c for c in range(1, sigma)], dtype=np.uint8)
    valid = list(reads[ok])
    doubled = []
    for r in valid:
        doubled += [r, comp[r[::-1]]]
    dsym, doff = synth.flatten(doubled)
    q = g.upload(vsym, voff, complement=comp)
    assert len(q) == 2 * len(valid)
    dexp = o.search_exact(dsym, doff)
    res = g.search_exact(q)
    assert hits_equal(strip_lb_rev(res.hits()), strip_lb_rev(dexp))
    assert locs_equal(g.locate(res).locs(), o.locate(dexp))


# ---- 4. k-error searches --------------------------------------------------------------------------------------------------------

@on_gpu(SCHEME_SIGMAS)
@pytest.mark.parametrize("edit", [False, True], ids=["hamming", "edit"])
@pytest.mark.parametrize("k", [1, 2])
def test_scheme_search(alpha, k, edit):
    from fmb200 import schemes
    from oracle.pyoracle import Counters
    o, g = alpha.o, alpha.g
    L = 32
    sym, off = _error_reads(alpha, 240, L, 50 + k, edit)
    sch = schemes.optimum(0, k)
    part = schemes.uniform_partition(sch[0].shape[1], L)
    ctr = Counters()
    exp = o.search_ng26(sym, off, sch, part, edit, counters=ctr)
    res = g.search_scheme(g.upload(sym, off), sch, part, edit)
    assert len(exp) > 0
    assert hits_equal(res.hits(), exp)
    assert locs_equal(g.locate(res).locs(), o.locate(exp))
    assert res.stats.extensions == ctr.extensions


def _same_list(got, exp):
    got, exp = np.asarray(got), np.asarray(exp)
    if got.shape != exp.shape:
        return False
    return all(np.array_equal(got[f].astype(np.uint64), exp[f].astype(np.uint64)) for f in ("qidx", "lb", "lb_rev", "len", "steps", "e"))


@on_gpu(SCHEME_SIGMAS)
@pytest.mark.parametrize("edit", [False, True], ids=["hamming", "edit"])
def test_search_n_in_order(alpha, edit):
    from fmb200 import schemes
    o, g = alpha.o, alpha.g
    L = 32
    sym, off = _error_reads(alpha, 240, L, 60, edit)
    q = g.upload(sym, off)
    for k in (1, 2):
        sch = schemes.optimum(0, k)
        part = schemes.uniform_partition(sch[0].shape[1], L)
        for n in (1, 3, 10**9):
            exp = o.search_ng26(sym, off, sch, part, edit, max_hits=n)
            assert len(exp) > 0
            assert _same_list(g.search_scheme(q, sch, part, edit, n=n).hits(), exp), (k, n)


@on_gpu(SCHEME_SIGMAS)
def test_pseudo_and_backtracking(alpha):
    from fmb200 import schemes
    o, g = alpha.o, alpha.g
    L = 24
    sym, off = _error_reads(alpha, 150, L, 70, True)
    sch = schemes.optimum(0, 1)
    part = schemes.uniform_partition(2, L)
    exp = o.search_pseudo(sym, off, schemes.expand(sch, part), True)
    assert len(exp) > 0
    assert hits_equal(g.search_scheme_pseudo(g.upload(sym, off), sch, part, True).hits(), exp)
    sym, off = _error_reads(alpha, 90, 12, 80, False)
    exp = o.search_backtracking(sym, off, 1)
    res = g.search_backtracking(g.upload(sym, off), 1)
    assert len(exp) > 0
    assert hits_equal(res.hits(), exp)
    assert locs_equal(g.locate(res).locs(), o.locate(exp))


@on_gpu([31, 32])
def test_k_error_search_is_refused_above_sigma_28(gpu, alpha):
    from fmb200 import schemes, synth
    g = alpha.g
    reads, _ = synth.reads_from_text(alpha.text[:LENGTHS[0] + 1], 8, 20, 1)
    q = g.upload(*synth.flatten(reads))
    sch, part = schemes.optimum(0, 1), schemes.uniform_partition(2, 20)
    for call in (lambda: g.search_scheme(q, sch, part, True), lambda: g.search_scheme(q, sch, part, False, n=3),
                 lambda: g.search_scheme_pseudo(q, sch, part, True), lambda: g.search_backtracking(q, 1)):
        with pytest.raises(gpu.FmbError) as e:
            call()
        assert e.value.code == FMB_EUNSUPPORTED


# ---- 5. where the discovery-order keys of the hit-limited search stop fitting ----------------------------------------------------

def key_bits(sigma, max_errors, length):
    """bits of one error slot of the discovery-order key (key_layout, csrc/fmb_search.cu): distances 0 .. length + 2 K + 2 plus an
    edge code per distance, 2 sigma + 2 kinds of edge; K slots of these bits must fit 56"""
    maxd = length + 2 * max_errors + 2
    values = maxd + 1 + maxd * (2 * sigma + 2)
    bits = 1
    while (1 << bits) < values:
        bits += 1
    return bits


def test_key_bits_worked_example():
    assert 4 * key_bits(28, 4, 267) == 56 and 4 * key_bits(28, 4, 268) == 60


@on_gpu([3, 16, 28])
def test_hit_limit_key_boundary(gpu, alpha):
    """a scheme with up to K = 4 errors (an exact half, then the errors): one symbol below the first query length whose keys need more
    than 56 bits the hit-limited search matches the oracle in order, at that length it is refused before any kernel runs"""
    from fmb200 import capi, synth
    sigma, o, g = alpha.sigma, alpha.o, alpha.g
    K = 4
    limit = next(L for L in range(2, 1 << 16) if K * key_bits(sigma, K, L) > 56)
    assert limit <= LENGTHS[0] // 2
    sch = (np.array([[0, 1]]), np.array([[0, 0]]), np.array([[0, K]]))
    for L in (limit - 1, limit):
        reads, _ = synth.reads_from_text(alpha.text[:LENGTHS[0] + 1], 40, L, L)
        part = [L // 2, L - L // 2]
        reads[20:, part[0]:] = synth.plant_errors(reads[20:, part[0]:], sigma, 2, False, 3)     # errors in the second part only
        sym, off = synth.flatten(reads)
        q = g.upload(sym, off)
        if L < limit:
            exp = o.search_ng26(sym, off, sch, part, False, max_hits=3)
            assert len(exp) >= 40
            assert _same_list(g.search_scheme(q, sch, part, False, n=3).hits(), exp)
        else:
            launches = capi.kernel_launch_count()
            with pytest.raises(gpu.FmbError) as e:
                g.search_scheme(q, sch, part, False, n=3)
            assert e.value.code == FMB_EUNSUPPORTED
            assert capi.kernel_launch_count() == launches


# ---- 6. extraction --------------------------------------------------------------------------------------------------------------

@on_gpu(SIGMAS)
def test_extract(alpha):
    seqs = _sequences(alpha.text)
    check_index(alpha.g, seqs, alpha.text, seed=alpha.sigma, count=2000)


@on_gpu([3, 12])
def test_extract_unidirectional(gpu, alpha):
    g = gpu.Index.build(alpha.sigma, alpha.text, sampling_rate=RATE, bidirectional=False)
    seqs = _sequences(alpha.text)
    check_index(g, seqs, alpha.text, seed=alpha.sigma + 1, count=2000)


# ---- 7. the oracle itself, without a GPU ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("sigma", SIGMAS)
def test_oracle_exact_counts_equal_substring_counts(sigma):
    """the oracle's exact-search rows of a pattern = the pattern's occurrences in the text, counted directly (patterns without the
    delimiter: within a sequence, and random ones over 1 .. sigma - 1)"""
    from numpy.lib.stride_tricks import sliding_window_view
    from fmb200 import synth
    text = synth.multi_text(LENGTHS, sigma, 40 + sigma)
    o = Oracle.build(text, sigma, RATE, True)
    rng = np.random.default_rng(sigma)
    pats = []
    for L in READ_LENGTHS:
        for _ in range(6):
            p = int(rng.integers(0, LENGTHS[0] - L))
            pats.append(text[p:p + L].copy())
    for L in range(1, 9):
        for _ in range(6):
            pats.append(rng.integers(1, sigma, size=L).astype(np.uint8))
    sym, off = synth.flatten(pats)
    hits = o.search_exact(sym, off)
    got = np.zeros(len(pats), dtype=np.int64)
    got[hits["qidx"].astype(np.int64)] = hits["len"].astype(np.int64)
    exp = np.array([int((sliding_window_view(text, p.size) == p).all(axis=1).sum()) for p in pats])
    assert np.array_equal(got, exp)
    assert exp.max() > 1
