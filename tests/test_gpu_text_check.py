"""Text check of exact search (FMB_TEXT_CHECK): once the interval of a read is one row, the rest of the read is compared with the text
at that row's position and the final row comes from the inverse suffix array; locate takes the position found there.  Hits, located
rows and lf_steps must equal the oracle's with the tables on and off (knob FMB_NO_TEXTCHECK, exact mode FMB_EXACT_NO_TEXT)."""
import os

import numpy as np
import pytest

from helpers import hits_equal, locs_equal, make_index_pair
from oracle.pyoracle import Counters, Oracle

pytestmark = pytest.mark.gpu

TEXT_CHECK, TEXT_LOCATE = 1, 2
NO_TEXT = 3


def _reads(text, seed):
    """reads of every kind the check meets: inside sequences, at their first / last symbol, across delimiters, random, with 0 / N"""
    rng = np.random.default_rng(seed)
    delim = np.flatnonzero(text == 0)
    starts = np.concatenate([[0], delim[:-1] + 1])
    reads = []
    for L in (15, 16, 17, 30, 40, 64, 100, 150, 300, 513, 700, 1100):
        if L >= text.size:
            continue
        for _ in range(30):
            p = int(rng.integers(0, text.size - L))
            reads.append(text[p:p + L].copy())                           # may straddle a delimiter
        for s, e in zip(starts, delim):
            if e - s >= L:
                reads.append(text[s:s + L].copy())                        # starts at position 0 of a sequence
                reads.append(text[e - L:e].copy())                        # ends at the last symbol of a sequence
        for _ in range(10):
            reads.append(rng.integers(1, 5, size=L).astype(np.uint8))      # random: does not occur
        for _ in range(5):
            r = text[int(rng.integers(0, text.size - L)):][:L].copy()
            r[int(rng.integers(0, L))] = int(rng.integers(0, 5))          # a symbol 0 (byte path) or a substitution
            reads.append(r)
            if L > 20:
                r = text[int(rng.integers(0, text.size - L)):][:L].copy()
                i = int(rng.integers(0, 4))
                r[i] = r[i] % 4 + 1 if r[i] else r[i]                     # mismatch in the first symbols: found late by the check
                reads.append(r)
    from fmb200 import synth
    return synth.flatten([r for r in reads if r.size])


def _check(g, o, sym, off, modes=(0, NO_TEXT)):
    exp = o.search_exact(sym, off)
    ctr = Counters()
    exp_locs = o.locate(exp, ctr)
    q = g.upload(sym, off)
    for mode in modes:
        g.set_exact_mode(mode)
        res = g.search_exact(q)
        loc = g.locate(res)
        assert hits_equal(res.hits(), exp), mode
        assert locs_equal(loc.locs(), exp_locs), mode
        assert loc.stats.lf_steps == ctr.lf_steps, mode
    g.set_exact_mode(0)


@pytest.mark.parametrize("lengths", [[40000], [3000, 1, 2, 700, 5, 129, 128, 127, 511, 512, 513, 2000], [300] * 50, [20] * 200 + [5000]])
def test_text_check_matches_oracle(gpu, lengths):
    from fmb200 import synth
    text = synth.multi_text(lengths, 5, 41)
    o, g = make_index_pair(gpu, text, 5, 4)
    assert g.info.text_tables == TEXT_CHECK | TEXT_LOCATE
    _check(g, o, *_reads(text, 3))


def test_single_rows_inside_the_kmer_table_and_repeats(gpu):
    """a 1 Mbp text (k-mer table of 14-mers: most reads are single rows after its lookup) with a repeated block (len > 1 hits)"""
    from fmb200 import synth
    base = synth.text(1 << 20, 5, 9)[:-1]
    rep = base[1000:1400].copy()
    text = np.concatenate([base[:200000], rep, base[200000:600000], rep, base[600000:], [0]]).astype(np.uint8)
    o, g = make_index_pair(gpu, text, 5, 16)
    assert g.info.text_tables == TEXT_CHECK | TEXT_LOCATE
    sym, off = _reads(text, 5)
    reads = [rep[i:i + 150] for i in range(0, 250, 10)]
    s2, o2 = synth.flatten(reads)
    sym = np.concatenate([sym, s2])
    off = np.concatenate([off, off[-1] + o2[1:]])
    _check(g, o, sym, off)


def test_knob_and_budget_leave_the_tables_out(gpu):
    from fmb200 import capi, synth
    text = synth.multi_text([30000, 700, 4000], 5, 17)
    o, g = make_index_pair(gpu, text, 5, 8)
    sym, off = _reads(text, 7)
    with_tables = g.info
    assert with_tables.text_tables == TEXT_CHECK | TEXT_LOCATE
    os.environ["FMB_NO_TEXTCHECK"] = "1"
    try:
        o2, g2 = make_index_pair(gpu, text, 5, 8)
    finally:
        del os.environ["FMB_NO_TEXTCHECK"]
    assert g2.info.text_tables == 0 and g2.info.tables == with_tables.tables
    n = text.size
    assert with_tables.device_bytes - g2.info.device_bytes >= 4 * n + n // 4
    _check(g2, o, sym, off, modes=(0,))
    try:
        for budget, want in ((g2.info.device_bytes + n, 0), (2 * with_tables.device_bytes, TEXT_CHECK | TEXT_LOCATE)):
            capi.set_image_budget(budget)
            _, g3 = make_index_pair(gpu, text, 5, 8)
            assert g3.info.text_tables == want
            _check(g3, o, sym, off, modes=(0,))
    finally:
        capi.set_image_budget(0)


def test_every_constructor_holds_the_same_tables(gpu, tmp_path):
    from fmb200 import synth
    text = synth.multi_text([9000, 300, 1, 2500], 5, 23)
    o = Oracle.build(text, 5, 4)
    built = gpu.Index.build(5, text, sampling_rate=4, device=0)
    bm, sq, sp = o.samples
    created = gpu.Index.from_bwt(5, o.bwt, o.bwt_rev, bm, sq, sp, device=0)
    path = str(tmp_path / "ix.fmb")
    built.save(path)
    loaded = gpu.Index.load(path, device=0)
    indices = [built, created, loaded]
    if gpu.device_count() > 1:
        indices.append(built.replicate(1))
    sym, off = _reads(text, 11)
    for g in indices:
        i = g.info
        assert i.text_tables == TEXT_CHECK | TEXT_LOCATE and i.device_bytes == built.info.device_bytes and i.tables == built.info.tables
        _check(g, o, sym, off)


def test_irregular_sampling_checks_reads_but_locates_by_the_table(gpu):
    """SA-space sampling of every 13th row: the check still decides the reads, locate keeps locrow + samples (lf_steps of the walk)"""
    from fmb200 import synth
    text = synth.multi_text([6000, 900], 5, 31)
    o = Oracle.build(text, 5, 4)
    sa = o.sa
    keep = np.zeros(text.size, dtype=bool)
    keep[::13] = True
    delim = np.flatnonzero(text == 0)
    seq_of = np.searchsorted(delim, sa[keep], side="left").astype(np.uint32)
    start = np.concatenate([[0], delim + 1])
    pos_of = (sa[keep] - start[seq_of]).astype(np.uint32)
    bm = np.zeros((text.size + 63) // 64, dtype=np.uint64)
    idx = np.flatnonzero(keep)
    np.bitwise_or.at(bm, idx // 64, np.uint64(1) << (idx % 64).astype(np.uint64))
    g = gpu.Index.from_bwt(5, o.bwt, o.bwt_rev, bm, seq_of, pos_of)
    o2 = Oracle.from_bwt(5, o.bwt, o.bwt_rev, bm, seq_of, pos_of)
    # walks that cross a delimiter leave no consistent row -> position map (no tables); either way locate keeps locrow + samples
    assert not g.info.text_tables & TEXT_LOCATE
    reads, _ = synth.reads_from_text(text[:6001], 300, 60, 4)
    sym, off = synth.flatten(reads)
    _check(g, o2, sym, off)


def test_line_requests_drop_with_the_check(gpu):
    """150-symbol reads of one long sequence: fewer requests per read with the check than with the LF jumps"""
    from fmb200 import synth
    text = synth.text(1 << 21, 5, 2)
    o, g = make_index_pair(gpu, text, 5, 16)
    reads, _ = synth.reads_from_text(text, 5000, 150, 8)
    sym, off = synth.flatten(reads)
    q = g.upload(sym, off)
    g.set_exact_mode(NO_TEXT)
    jumps = g.search_exact(q).stats.line_requests
    g.set_exact_mode(0)
    check = g.search_exact(q).stats.line_requests
    assert check < jumps
