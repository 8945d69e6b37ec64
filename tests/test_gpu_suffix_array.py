"""Suffix array in place of the locate shortcut (DNA layout, text-regular sampling): sa[row] = text position of the row's suffix, one
fetch per located row, the sequence found through the per-4096-symbol block table.  Every row must locate to the oracle's suffix array;
hits, located rows and lf_steps must be identical with the suffix array and with the shortcut it replaces (knob FMB_NO_SA)."""
import os

import numpy as np
import pytest

from helpers import hits_equal, locs_equal, make_index_pair
from oracle.pyoracle import Counters, Oracle

pytestmark = pytest.mark.gpu

LOCROW = 32
TEXT_CHECK, TEXT_LOCATE = 1, 2
NO_TEXT = 3
RATE = 16

COLLECTIONS = {
    "one_sequence": [50000],
    # several sequences start inside one 4096-symbol block (and some at its first symbols), next to long ones
    "many_short": [3000, 1, 2, 700, 5, 129, 128, 127, 511, 512, 513, 2000] + [37] * 300 + [9000],
    # sequences shorter than the sampling rate, the first one among them
    "shorter_than_rate": [9, 3, 1, 20000, 2, 15, 14, 16, 17, 6000],
}


def _without_sa(make):
    os.environ["FMB_NO_SA"] = "1"
    try:
        return make()
    finally:
        del os.environ["FMB_NO_SA"]


def _text(lengths, seed=41):
    from fmb200 import synth
    return synth.multi_text(lengths, 5, seed)


def _seq_pos(text, g):
    """(seq, pos) of global text positions g of s0 0 s1 0 ..."""
    delim = np.flatnonzero(text == 0)
    start = np.concatenate([[0], delim[:-1] + 1]).astype(np.int64)
    g = np.asarray(g, dtype=np.int64)
    seq = np.searchsorted(start, g, side="right") - 1
    return seq.astype(np.uint32), (g - start[seq]).astype(np.uint32)


def _every_row(g):
    """located rows of the queries "0" .. "4": their intervals tile all rows in order, so the i-th located row is row i"""
    from fmb200 import synth
    sym, off = synth.flatten([np.array([c], dtype=np.uint8) for c in range(5)])
    res = g.search_exact(g.upload(sym, off))
    loc = g.locate(res)
    return loc.locs(), loc.stats.lf_steps


def _oracle_steps(o):
    from fmb200 import synth
    sym, off = synth.flatten([np.array([c], dtype=np.uint8) for c in range(5)])
    ctr = Counters()
    o.locate(o.search_exact(sym, off), ctr)
    return ctr.lf_steps


@pytest.mark.parametrize("name", list(COLLECTIONS))
def test_every_row_locates_to_the_oracle_suffix_array(gpu, name):
    text = _text(COLLECTIONS[name])
    o, g = make_index_pair(gpu, text, 5, RATE)
    _, g2 = _without_sa(lambda: make_index_pair(gpu, text, 5, RATE))
    assert g.info.tables & LOCROW and g2.info.tables == g.info.tables
    assert g.info.text_tables == g2.info.text_tables == TEXT_CHECK | TEXT_LOCATE
    # the suffix array takes the shortcut's 4 bytes per row; the sequence table adds 8 bytes per 4096 symbols
    assert g.info.device_bytes - g2.info.device_bytes == 8 * ((text.size >> 12) + 2)
    locs, steps = _every_row(g)
    locs2, steps2 = _every_row(g2)
    seq, pos = _seq_pos(text, o.sa)
    assert locs.size == text.size
    assert np.array_equal(locs["seq"], seq) and np.array_equal(locs["pos"], pos)
    assert np.array_equal(locs, locs2)
    assert steps == steps2 == _oracle_steps(o)


def test_built_created_and_loaded_indices_agree(gpu, tmp_path):
    text = _text(COLLECTIONS["many_short"], 23)
    o = Oracle.build(text, 5, RATE)
    built = gpu.Index.build(5, text, sampling_rate=RATE, device=0)
    bm, sq, sp = o.samples
    created = gpu.Index.from_bwt(5, o.bwt, o.bwt_rev, bm, sq, sp, device=0)
    path = str(tmp_path / "ix.fmb")
    built.save(path)
    loaded = gpu.Index.load(path, device=0)
    seq, pos = _seq_pos(text, o.sa)
    want_steps = _oracle_steps(o)
    for g in (built, created, loaded):
        assert g.info.device_bytes == built.info.device_bytes and g.info.tables == built.info.tables
        locs, steps = _every_row(g)
        assert np.array_equal(locs["seq"], seq) and np.array_equal(locs["pos"], pos)
        assert steps == want_steps


def _reads(text, seed):
    """reads inside sequences, at their first / last symbols, across delimiters, random, and reads whose last symbols start a sequence
    while the first ones do not precede it in the text (they would start before their sequence)"""
    from fmb200 import synth
    rng = np.random.default_rng(seed)
    delim = np.flatnonzero(text == 0)
    starts = np.concatenate([[0], delim[:-1] + 1])
    reads = []
    for L in (16, 17, 40, 100, 150, 300):
        for _ in range(40):
            p = int(rng.integers(0, text.size - L))
            reads.append(text[p:p + L].copy())
        for s, e in zip(starts, delim):
            if e - s >= L:
                reads.append(text[s:s + L].copy())
                reads.append(text[e - L:e].copy())
                head = rng.integers(1, 5, size=20).astype(np.uint8)
                reads.append(np.concatenate([head, text[s:s + L]]))
        for _ in range(10):
            reads.append(rng.integers(1, 5, size=L).astype(np.uint8))
    return synth.flatten(reads)


@pytest.mark.parametrize("name", list(COLLECTIONS))
def test_exact_hits_and_located_rows_with_and_without_sa(gpu, name):
    text = _text(COLLECTIONS[name], 7)
    o, g = make_index_pair(gpu, text, 5, RATE)
    _, g2 = _without_sa(lambda: make_index_pair(gpu, text, 5, RATE))
    sym, off = _reads(text, 3)
    exp = o.search_exact(sym, off)
    ctr = Counters()
    exp_locs = o.locate(exp, ctr)
    for index in (g, g2):
        q = index.upload(sym, off)
        for mode in (0, NO_TEXT):
            index.set_exact_mode(mode)
            res = index.search_exact(q)
            loc = index.locate(res)
            assert hits_equal(res.hits(), exp), mode
            assert locs_equal(loc.locs(), exp_locs), mode
            assert loc.stats.lf_steps == ctr.lf_steps, mode
        index.set_exact_mode(0)


def test_k_error_locate_with_and_without_sa(gpu):
    from fmb200 import schemes, synth
    text = _text(COLLECTIONS["many_short"], 13)
    o, g = make_index_pair(gpu, text, 5, RATE)
    _, g2 = _without_sa(lambda: make_index_pair(gpu, text, 5, RATE))
    reads, _ = synth.reads_from_text(text[:3001], 400, 60, 5)
    reads = synth.plant_errors(reads, 5, 1, True, 6)
    sym, off = synth.flatten(reads)
    sch, part = schemes.optimum(0, 1), schemes.uniform_partition(2, 60)
    exp = o.search_ng26(sym, off, sch, part, True)
    ctr = Counters()
    exp_locs = o.locate(exp, ctr)
    for index in (g, g2):
        loc = index.locate(index.search_scheme(index.upload(sym, off), sch, part, True))
        assert locs_equal(loc.locs(), exp_locs)
        assert loc.stats.lf_steps == ctr.lf_steps


def test_line_requests_drop_by_one_per_checked_read(gpu):
    """150-symbol reads of one long sequence: the suffix array replaces two dependent requests (shortcut word, sample) by one"""
    from fmb200 import synth
    text = synth.text(1 << 21, 5, 2)
    _, g = make_index_pair(gpu, text, 5, RATE)
    _, g2 = _without_sa(lambda: make_index_pair(gpu, text, 5, RATE))
    reads, _ = synth.reads_from_text(text, 5000, 150, 8)
    sym, off = synth.flatten(reads)
    res = g.search_exact(g.upload(sym, off))
    res2 = g2.search_exact(g2.upload(sym, off))
    assert hits_equal(res.hits(), res2.hits())
    checked = int(np.count_nonzero(res.hits()["len"] == 1))
    assert checked > 4000
    assert res2.stats.line_requests - res.stats.line_requests >= checked


def test_irregular_sampling_keeps_the_shortcut(gpu):
    """SA-space sampling of every 13th row: lf_steps are those of the walk, so locate keeps the shortcut (no sequence table)"""
    from fmb200 import synth
    text = synth.multi_text([6000, 900], 5, 31)
    o = Oracle.build(text, 5, 4)
    keep = np.zeros(text.size, dtype=bool)
    keep[::13] = True
    seq_of, pos_of = _seq_pos(text, o.sa[keep])
    bm = np.zeros((text.size + 63) // 64, dtype=np.uint64)
    idx = np.flatnonzero(keep)
    np.bitwise_or.at(bm, idx // 64, np.uint64(1) << (idx % 64).astype(np.uint64))
    g = gpu.Index.from_bwt(5, o.bwt, o.bwt_rev, bm, seq_of, pos_of)
    g2 = _without_sa(lambda: gpu.Index.from_bwt(5, o.bwt, o.bwt_rev, bm, seq_of, pos_of))
    o2 = Oracle.from_bwt(5, o.bwt, o.bwt_rev, bm, seq_of, pos_of)
    assert g.info.tables & LOCROW and not g.info.text_tables & TEXT_LOCATE
    assert g.info.device_bytes == g2.info.device_bytes
    reads, _ = synth.reads_from_text(text[:6001], 300, 60, 4)
    sym, off = synth.flatten(reads)
    exp = o2.search_exact(sym, off)
    ctr = Counters()
    exp_locs = o2.locate(exp, ctr)
    loc = g.locate(g.search_exact(g.upload(sym, off)))
    assert locs_equal(loc.locs(), exp_locs) and loc.stats.lf_steps == ctr.lf_steps
