"""Every locate path against the oracle: the same exact and k = 1 hits located through the suffix array, the shortcut word, the lane-pair
walk on the locate blocks and the one-thread walk, on both occurrence layouts and with irregular sampling, each also in FMB_LOCATE_WALK
mode.  Located rows, lf_steps and locate_rows (seq, pos, steps) must equal the oracle's; the image's tables pin the path each case
takes."""
import os

import numpy as np
import pytest

from helpers import hits_equal, locs_equal, make_index_pair
from oracle.pyoracle import Counters, Oracle

pytestmark = pytest.mark.gpu

LOCBLOCK, LOCROW = 16, 32
TEXT_CHECK, TEXT_LOCATE = 1, 2
RATE = 16
WALK = 1

# case: (sigma, knobs, tables & (LOCBLOCK | LOCROW), text_tables)
CASES = {
    "dna_sa": (5, (), LOCBLOCK | LOCROW, TEXT_CHECK | TEXT_LOCATE),
    "dna_shortcut": (5, ("FMB_NO_SA",), LOCBLOCK | LOCROW, TEXT_CHECK | TEXT_LOCATE),
    "dna_pair_walk": (5, ("FMB_NO_LOCROW",), LOCBLOCK, 0),
    "dna_thread_walk": (5, ("FMB_NO_LOCBLOCKS",), 0, 0),
    "dna_irregular": (5, (), LOCBLOCK | LOCROW, None),
    "gen_shortcut": (21, (), LOCROW, 0),
    "gen_walk": (21, ("FMB_NO_LOCROW",), 0, 0),
}
_BUILT = {}


def _collection(sigma, seed=5):
    """short and long sequences; a 300-symbol unit copied into several of them, so that reads of it have multi-row intervals"""
    from fmb200 import synth
    lengths = [3000, 5, 1, 700, 129, 16, 2000] + [37] * 40 + [1500, 1200]
    seqs = [synth.text(n + 1, sigma, seed + 7919 * k)[:-1] for k, n in enumerate(lengths)]
    unit = seqs[0][100:400].copy()
    for k, at in ((3, 50), (6, 900), (6, 1500), (47, 0), (48, 700)):
        seqs[k][at:at + unit.size] = unit
    return seqs, np.concatenate([np.append(s, 0).astype(np.uint8) for s in seqs])


def _irregular(gpu, text, sigma, every=13):
    """fmb_index_create with every 13th row sampled: walks of up to ~100 steps, lf_steps no longer pos % rate"""
    o = Oracle.build(text, sigma, 4)
    keep = np.zeros(text.size, dtype=bool)
    keep[::every] = True
    delim = np.flatnonzero(text == 0)
    start = np.concatenate([[0], delim[:-1] + 1])
    g = o.sa[keep].astype(np.int64)
    seq = (np.searchsorted(start, g, side="right") - 1).astype(np.uint32)
    pos = (g - start[seq]).astype(np.uint32)
    bm = np.zeros((text.size + 63) // 64, dtype=np.uint64)
    idx = np.flatnonzero(keep)
    np.bitwise_or.at(bm, idx // 64, np.uint64(1) << (idx % 64).astype(np.uint64))
    return Oracle.from_bwt(sigma, o.bwt, o.bwt_rev, bm, seq, pos), gpu.Index.from_bwt(sigma, o.bwt, o.bwt_rev, bm, seq, pos)


def _case(gpu, name):
    if name not in _BUILT:
        sigma, knobs, _, _ = CASES[name]
        seqs, text = _collection(sigma)
        for k in knobs:
            os.environ[k] = "1"
        try:
            o, g = _irregular(gpu, text, sigma) if name == "dna_irregular" else make_index_pair(gpu, text, sigma, RATE)
        finally:
            for k in knobs:
                del os.environ[k]
        _BUILT[name] = (seqs, text, o, g)
    return _BUILT[name]


def _exact_reads(seqs, sigma, seed):
    """windows of 8 .. 100 symbols inside sequences (unique ones: single rows the text check takes; in the unit: several rows) and
    random reads"""
    from fmb200 import synth
    rng = np.random.default_rng(seed)
    reads = []
    for L in (8, 20, 40, 100):
        reads += [seqs[0][p:p + L].copy() for p in (100, 150)]
        for s in seqs:
            if s.size >= L:
                for _ in range(4):
                    p = int(rng.integers(0, s.size - L + 1))
                    reads.append(s[p:p + L].copy())
        reads += [rng.integers(1, sigma, size=L).astype(np.uint8) for _ in range(10)]
    return synth.flatten(reads)


def _k1_reads(text, sigma, seed):
    from fmb200 import synth
    reads, _ = synth.reads_from_text(text[:3001], 300, 40, seed)
    return synth.flatten(synth.plant_errors(reads, sigma, 1, True, seed + 1))


@pytest.mark.parametrize("walk", [False, True])
@pytest.mark.parametrize("name", list(CASES))
def test_every_locate_path_against_oracle(gpu, name, walk):
    from fmb200 import schemes
    sigma, _, tables, text_tables = CASES[name]
    seqs, text, o, g = _case(gpu, name)
    info = g.info
    assert info.tables & (LOCBLOCK | LOCROW) == tables
    if text_tables is None:
        assert not info.text_tables & TEXT_LOCATE
    else:
        assert info.text_tables == text_tables
    if name == "dna_sa":
        # the suffix array in place of the shortcut: only the per-4096-symbol sequence table differs
        assert info.device_bytes - _case(gpu, "dna_shortcut")[3].info.device_bytes == 8 * ((text.size >> 12) + 2)
    g.set_locate_mode(WALK if walk else 0)
    try:
        sym, off = _exact_reads(seqs, sigma, 3)
        exp = o.search_exact(sym, off)
        assert (exp["len"] == 1).any() and (exp["len"] > 1).any()
        ctr = Counters()
        exp_locs = o.locate(exp, ctr)
        res = g.search_exact(g.upload(sym, off))
        assert hits_equal(res.hits(), exp)
        loc = g.locate(res)
        assert locs_equal(loc.locs(), exp_locs) and loc.stats.lf_steps == ctr.lf_steps

        sym, off = _k1_reads(text, sigma, 11)
        sch, part = schemes.optimum(0, 1), schemes.uniform_partition(2, 40)
        exp = o.search_ng26(sym, off, sch, part, True)
        ctr = Counters()
        exp_locs = o.locate(exp, ctr)
        loc = g.locate(g.search_scheme(g.upload(sym, off), sch, part, True))
        assert locs_equal(loc.locs(), exp_locs) and loc.stats.lf_steps == ctr.lf_steps
    finally:
        g.set_locate_mode(0)
    rows = np.arange(0, text.size, 7, dtype=np.uint64)
    seq, pos, steps = g.locate_rows(rows)
    want = np.array([o.locate_row(int(r)) for r in rows], dtype=np.uint64).reshape(-1, 3)
    assert np.array_equal(seq, want[:, 0]) and np.array_equal(pos, want[:, 1]) and np.array_equal(steps, want[:, 2])
