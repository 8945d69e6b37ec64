"""Super-maximal exact matches (fmb_search_smems, fmb_locate_smems): records and located rows equal an oracle written from the
definition alone (substring search over the sequences, no FM code), on both occurrence layouts, every table configuration and sampling
the library accepts; the work counter equals the reference algorithm's; the refusals launch nothing; and at scale every SMEM passes
the certificate of tools/smem_certificate.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import Oracle
from tools.smem_certificate import certify

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U64MAX = (1 << 64) - 1
FMB_TABLE_BIKMER = 64


# ---- oracle from the definition -------------------------------------------------------------------------------------------------
def smems_by_definition(seqs, sigma, query):
    """[i, e[i]) for every i with e[i] > i and (i == 0 or e[i-1] < e[i]); e[i] = end of the longest occurring stretch from i"""
    hay = [bytes(np.asarray(s, dtype=np.uint8)) for s in seqs]
    q = np.asarray(query, dtype=np.uint8)
    m = q.size
    ok = (q >= 1) & (q < sigma)

    def occurs(i, j):
        if not ok[i:j].all():
            return False
        needle = bytes(q[i:j])
        return any(needle in h for h in hay)

    e = np.zeros(m, dtype=np.int64)
    j = 0
    for i in range(m):
        j = max(j, i)
        while j < m and occurs(i, j + 1):
            j += 1
        e[i] = j
    return [(i, int(e[i])) for i in range(m) if e[i] > i and (i == 0 or e[i - 1] < e[i])]


def oracle_smems(o, seqs, sigma, queries, min_len=0):
    """records (qidx, begin, end, lb, len), ordered by qidx then begin; intervals from Oracle.search_exact"""
    recs = [(qi, b, e) for qi, qs in enumerate(queries) for b, e in smems_by_definition(seqs, sigma, qs) if e - b >= max(min_len, 1)]
    out = np.zeros(len(recs), dtype=[("qidx", "<u8"), ("begin", "<u8"), ("end", "<u8"), ("lb", "<u8"), ("len", "<u8")])
    if not recs:
        return out
    subs = [np.asarray(queries[qi][b:e], dtype=np.uint8) for qi, b, e in recs]
    off = np.zeros(len(subs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([s.size for s in subs])
    h = o.search_exact(np.concatenate(subs), off)
    lb = np.zeros(len(recs), dtype=np.uint64)
    ln = np.zeros(len(recs), dtype=np.uint64)
    lb[h["qidx"].astype(np.int64)], ln[h["qidx"].astype(np.int64)] = h["lb"], h["len"]
    assert (ln > 0).all()
    out["qidx"], out["begin"], out["end"] = zip(*recs)
    out["lb"], out["len"] = lb, ln
    return out


def oracle_locs(o, recs, max_occ=None):
    """Oracle.locate of the rows lb .. lb + min(len, max_occ) - 1 of every record, grouped by record, in row order"""
    cap = U64MAX if max_occ is None else max_occ
    hits = np.zeros(recs.size, dtype=[("qidx", "<u8"), ("lb", "<u8"), ("lb_rev", "<u8"), ("len", "<u8"), ("steps", "<u8"), ("e", "<u8")])
    hits["qidx"] = np.arange(recs.size)
    hits["lb"] = recs["lb"]
    hits["len"] = np.minimum(recs["len"], np.uint64(cap))
    locs = o.locate(hits)
    r = recs[locs["qidx"].astype(np.int64)]
    out = np.zeros(locs.size, dtype=[("qidx", "<u8"), ("begin", "<u8"), ("end", "<u8"), ("seq", "<u8"), ("pos", "<u8")])
    out["qidx"], out["begin"], out["end"] = r["qidx"], r["begin"], r["end"]
    out["seq"], out["pos"] = locs["seq"], locs["pos"]
    return out


def reference_algorithm(o, sigma, query, min_len=0):
    """the SMEM algorithm of the library on Oracle.extend: (records (begin, end, lb, len), extensions)"""
    q = [int(c) for c in query]
    m = len(q)
    whole = np.array([0, 0, o.n, 0], dtype=np.uint64)
    ok = lambda c: 1 <= c < sigma  # noqa: E731
    out, ext = [], 0
    x, j, cur = 0, 0, None
    while x < m:
        if cur is None:
            if not ok(q[x]):
                x += 1
                continue
            cur = o.extend(whole, q[x], True); ext += 1
            if cur[2] == 0:
                x += 1; cur = None
                continue
            j = x + 1
        while j < m and ok(q[j]):
            nxt = o.extend(cur, q[j], True); ext += 1
            if nxt[2] == 0:
                break
            cur = nxt; j += 1
        if j - x >= max(min_len, 1):
            out.append((x, j, int(cur[0]), int(cur[2])))
        if j == m:
            break
        if not ok(q[j]):
            x = j + 1; cur = None
            continue
        cur = o.extend(whole, q[j], False); ext += 1
        if cur[2] == 0:
            x = j + 1; cur = None
            continue
        b = j
        while b - 1 > x and ok(q[b - 1]):
            nxt = o.extend(cur, q[b - 1], False); ext += 1
            if nxt[2] == 0:
                break
            cur = nxt; b -= 1
        x = b; j = j + 1
    return out, ext


# ---- workloads ------------------------------------------------------------------------------------------------------------------
def collection(kind, sigma, seed):
    rng = np.random.default_rng(seed)
    if kind == "short":
        seqs = [rng.integers(1, sigma, size=int(rng.integers(1, 60)), dtype=np.uint8) for _ in range(150)]
    elif kind == "long":
        seqs = [rng.integers(1, sigma, size=int(rng.integers(1500, 3000)), dtype=np.uint8) for _ in range(3)]
    else:  # repetitive: copies of one unit with a few substitutions -> wide intervals
        unit = rng.integers(1, sigma, size=120, dtype=np.uint8)
        seqs = []
        for _ in range(30):
            s = unit.copy()
            k = rng.integers(0, s.size, size=2)
            s[k] = rng.integers(1, sigma, size=2)
            seqs.append(np.concatenate([rng.integers(1, sigma, size=int(rng.integers(0, 20)), dtype=np.uint8), s]))
    text = np.concatenate([np.append(s, np.uint8(0)) for s in seqs]).astype(np.uint8)
    return seqs, text


def make_queries(seqs, sigma, count, seed, length=(1, 70)):
    """windows of the sequences with substitutions, windows across sequence borders, random strings, symbols 0 / >= sigma"""
    rng = np.random.default_rng(seed)
    text = np.concatenate([np.append(s, np.uint8(0)) for s in seqs])
    out = []
    for i in range(count):
        L = int(rng.integers(*length))
        kind = i % 4
        if kind == 0 or kind == 1:
            s = seqs[int(rng.integers(len(seqs)))]
            p = int(rng.integers(0, max(1, s.size - L + 1)))
            r = s[p:p + L].copy()
            for _ in range(int(rng.integers(0, 4))):
                if r.size:
                    r[int(rng.integers(r.size))] = int(rng.integers(1, sigma))
        elif kind == 2:
            p = int(rng.integers(0, max(1, text.size - L)))
            r = text[p:p + L].copy()                     # may hold delimiters (symbol 0) and span sequences
        else:
            r = rng.integers(1, sigma, size=L).astype(np.uint8)
        if r.size and rng.random() < 0.15:
            r[int(rng.integers(r.size))] = rng.choice([0, sigma, 255])
        out.append(r.astype(np.uint8))
    return out


def flat(queries):
    off = np.zeros(len(queries) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(q) for q in queries])
    sym = np.concatenate([np.asarray(q, dtype=np.uint8) for q in queries]) if off[-1] else np.zeros(0, dtype=np.uint8)
    return sym, off


def gpu_smems(index, queries, min_len=0, **upload):
    sym, off = flat(queries)
    q = index.upload(sym, off, **upload)
    r = index.search_smems(q, min_len=min_len)
    assert r.kind == 2
    return r, r.smems()


def check_against_oracle(index, o, seqs, sigma, queries, min_lens=(0, 1, 19, 10**6), max_occs=(1, 3, None)):
    want = oracle_smems(o, seqs, sigma, queries)
    for ml in min_lens:
        r, got = gpu_smems(index, queries, ml)
        sel = want[(want["end"] - want["begin"]) >= max(ml, 1)]
        assert np.array_equal(got, sel), (ml, got.size, sel.size)
        if ml == 0:
            for mo in max_occs:
                lr = index.locate_smems(r, max_occ=mo)
                assert lr.kind == 3
                assert np.array_equal(lr.smem_locs(), oracle_locs(o, want, mo)), mo
    return want


# ---- the oracle itself ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sigma", [2, 5, 21])
def test_reference_algorithm_equals_definition(sigma):
    """the library's algorithm on Oracle.extend finds exactly the SMEMs of the definition"""
    seqs, text = collection("short", sigma, 3)
    o = Oracle.build(text, sigma, 4, True)
    for qs in make_queries(seqs, sigma, 80, 4):
        got, _ = reference_algorithm(o, sigma, qs)
        assert [(b, e) for b, e, _, _ in got] == smems_by_definition(seqs, sigma, qs)


# ---- records and rows against the oracle -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["short", "long", "repeat"])
@pytest.mark.parametrize("sigma", [2, 4, 5, 6, 21, 32])
def test_against_oracle(gpu, sigma, kind):
    seqs, text = collection(kind, sigma, 10 + sigma)
    index = gpu.Index.build(sigma, text, sampling_rate=4)
    o = Oracle.build(text, sigma, 4, True)
    queries = make_queries(seqs, sigma, 160, 20 + sigma)
    check_against_oracle(index, o, seqs, sigma, queries)
    if sigma == 5:
        assert index.info.text_tables & 1                    # the text path ran on this image
        r, _ = gpu_smems(index, queries)
        assert r.stats.line_requests > 0


@pytest.mark.parametrize("knobs", [("FMB_NO_BIKMER",), ("FMB_NO_TEXTCHECK",), ("FMB_NO_JUMP",), ("FMB_NO_SA",),
                                   ("FMB_NO_BIKMER", "FMB_NO_TEXTCHECK", "FMB_NO_JUMP")])
@pytest.mark.parametrize("sigma", [5, 21])
def test_table_knobs(gpu, monkeypatch, sigma, knobs):
    seqs, text = collection("long", sigma, 40 + sigma)
    for k in knobs:
        monkeypatch.setenv(k, "1")
    index = gpu.Index.build(sigma, text, sampling_rate=4)
    for k in knobs:
        monkeypatch.delenv(k)
    info = index.info
    if "FMB_NO_BIKMER" in knobs:
        assert not info.tables & FMB_TABLE_BIKMER
    if "FMB_NO_TEXTCHECK" in knobs:
        assert not info.text_tables & 1
    o = Oracle.build(text, sigma, 4, True)
    queries = make_queries(seqs, sigma, 120, 50 + sigma)
    check_against_oracle(index, o, seqs, sigma, queries, min_lens=(0, 19))
    if len(knobs) == 3:
        r, _ = gpu_smems(index, queries)
        assert r.stats.extensions == sum(reference_algorithm(o, sigma, qs)[1] for qs in queries)
        assert r.stats.line_requests == 0


def row_sampled_index(gpu, text, sigma, every=2):
    """fmb_index_create from BWT + samples taken every `every` rows (position 0 of a sequence is not always sampled)"""
    full = Oracle.build(text, sigma, 1, True)
    sa = np.asarray(full.sa, dtype=np.int64)
    delims = np.flatnonzero(text == 0)
    rows = np.arange(0, sa.size, every)
    p = sa[rows]
    seq = np.searchsorted(delims, p, side="left")
    pos = p - np.where(seq > 0, delims[np.maximum(seq - 1, 0)] + 1, 0)
    bits = np.zeros(sa.size, dtype=bool)
    bits[rows] = True
    packed = np.packbits(bits, bitorder="little")
    bm = np.concatenate([packed, np.zeros((-packed.size) % 8, dtype=np.uint8)]).view("<u8")
    seq, pos = seq.astype(np.uint32), pos.astype(np.uint32)
    # the oracle over the same BWT and samples: a locate walk that crosses a delimiter reports what the reference reports
    o = Oracle.from_bwt(sigma, full.bwt, full.bwt_rev, bm, seq, pos)
    return gpu.Index.from_bwt(sigma, full.bwt, full.bwt_rev, bm, seq, pos), o


@pytest.mark.parametrize("sigma", [5, 21])
def test_row_sampled_built_and_loaded_indices(gpu, tmp_path, sigma):
    seqs, text = collection("short", sigma, 60 + sigma)
    queries = make_queries(seqs, sigma, 120, 61 + sigma)
    index, o = row_sampled_index(gpu, text, sigma)
    check_against_oracle(index, o, seqs, sigma, queries, min_lens=(0,))
    built = gpu.Index.build(sigma, text, sampling_rate=8)
    o = Oracle.build(text, sigma, 8, True)
    check_against_oracle(built, o, seqs, sigma, queries, min_lens=(0,))
    path = str(tmp_path / "ix.fmb")
    built.save(path)
    check_against_oracle(gpu.Index.load(path), o, seqs, sigma, queries, min_lens=(0,))


# ---- edge cases ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dna(gpu):
    seqs, text = collection("long", 5, 77)
    return seqs, text, gpu.Index.build(5, text, sampling_rate=4), Oracle.build(text, 5, 4, True)


def expect(dna, queries):
    seqs, _, index, o = dna
    return check_against_oracle(index, o, seqs, 5, queries, min_lens=(0,), max_occs=(None,))


def test_exact_reads_one_smem(dna):
    seqs = dna[0]
    queries = [seqs[0][10:160], seqs[1][:150], seqs[2][-150:], seqs[0][500:517]]
    want = expect(dna, queries)
    assert want.size == 4 and (want["begin"] == 0).all() and np.array_equal(want["end"], [len(q) for q in queries])


def test_read_spanning_two_sequences_is_split(dna):
    seqs, text = dna[0], dna[1]
    border = len(seqs[0])                                  # the delimiter after sequence 0
    tail, head = seqs[0][-40:], seqs[1][:40]
    queries = [np.concatenate([tail, head]), text[border - 30:border + 31].copy()]
    want = expect(dna, queries)
    assert (want[want["qidx"] == 0]["end"] <= 40).any() and (want[want["qidx"] == 0]["begin"] >= 40).any()


def test_reads_running_past_sequence_ends(dna):
    seqs = dna[0]
    rng = np.random.default_rng(3)
    queries = [np.concatenate([rng.integers(1, 5, 30).astype(np.uint8), seqs[1][:50]]),
               np.concatenate([seqs[2][-50:], rng.integers(1, 5, 30).astype(np.uint8)])]
    expect(dna, queries)


def test_non_matching_and_absent_symbols(gpu):
    # sigma 5 index over symbols 1..3 only: symbol 4 has a code but occurs nowhere
    rng = np.random.default_rng(5)
    seqs = [rng.integers(1, 4, size=400).astype(np.uint8) for _ in range(4)]
    text = np.concatenate([np.append(s, np.uint8(0)) for s in seqs])
    index, o = gpu.Index.build(5, text, sampling_rate=4), Oracle.build(text, 5, 4, True)
    base = seqs[1][20:80]
    queries = []
    for bad in (0, 4, 5, 200):
        for at in (0, 30, base.size - 1):
            r = base.copy()
            r[at] = bad
            queries.append(r)
    check_against_oracle(index, o, seqs, 5, queries, min_lens=(0,), max_occs=(None,))


def test_query_lengths_zero_one_and_longer_than_every_sequence(dna):
    seqs = dna[0]
    longest = max(len(s) for s in seqs)
    queries = [np.zeros(0, dtype=np.uint8), seqs[0][:1], np.array([0], dtype=np.uint8), np.array([7], dtype=np.uint8),
               np.concatenate([seqs[0], seqs[1]])[: longest + 100]]
    want = expect(dna, queries)
    assert not (want["qidx"] == 0).any() and (want["qidx"] == 1).sum() == 1


def test_mixed_lengths(dna):
    seqs = dna[0]
    expect(dna, make_queries(seqs, 5, 200, 9, length=(0, 300)))


def test_revcomp_and_packed_uploads(gpu, dna):
    seqs, _, index, _ = dna
    queries = make_queries(seqs, 5, 200, 11, length=(20, 120))
    comp = np.array([0, 4, 3, 2, 1], dtype=np.uint8)
    both = []
    for qs in queries:
        rc = qs[::-1].copy()
        m = rc < 5
        rc[m] = comp[rc[m]]
        both += [qs, rc]
    _, explicit = gpu_smems(index, both)
    _, doubled = gpu_smems(index, queries, complement=comp)
    assert np.array_equal(doubled, explicit)
    sym, _ = flat(queries)
    _, packed = gpu_smems(index, queries, packed=gpu.capi.pack_queries(sym))
    _, plain = gpu_smems(index, queries)
    assert np.array_equal(packed, plain)


def test_split_uploads_equal_one_batch(dna):
    seqs, _, index, _ = dna
    queries = make_queries(seqs, 5, 300, 13)
    _, whole = gpu_smems(index, queries)
    parts = []
    for lo in range(0, len(queries), 70):
        _, p = gpu_smems(index, queries[lo:lo + 70])
        p["qidx"] += lo
        parts.append(p)
    assert np.array_equal(np.concatenate(parts), whole)


def test_record_list_grows(gpu):
    """random 40-symbol reads on a 1 Mbp text: about 30 SMEMs each, far beyond the first reservation of 2^20 records"""
    from fmb200 import capi
    n = 1_000_000
    d_text = capi.synth_text_device(0, 5, n, 21)
    try:
        index = gpu.Index.build_from_device_text(5, d_text, n, sampling_rate=16)
    finally:
        capi.device_free(0, d_text)
    rng = np.random.default_rng(2)
    nq, L = 200_000, 40
    sym = rng.integers(1, 5, size=nq * L).astype(np.uint8)
    off = np.arange(nq + 1, dtype=np.uint64) * np.uint64(L)
    whole = index.search_smems(index.upload(sym, off), min_len=0).smems()
    assert whole.size > (1 << 20)
    parts = []
    for lo in range(0, nq, 20_000):
        p = index.search_smems(index.upload(sym, off[lo:lo + 20_001]), min_len=0).smems()
        p["qidx"] += lo
        parts.append(p)
    assert np.array_equal(np.concatenate(parts), whole)
    assert certify(index, sym, off[:2001], whole[whole["qidx"] < 2000])


# ---- refusals --------------------------------------------------------------------------------------------------------------------------
def test_refusals_launch_nothing(gpu, dna):
    from fmb200 import capi
    L = capi.lib()
    seqs, text, index, o = dna
    queries = make_queries(seqs, 5, 20, 15)
    sym, off = flat(queries)
    q = index.upload(sym, off)
    hits = index.search_exact(q)
    smems = index.search_smems(q)
    uni = gpu.Index.build(5, text, sampling_rate=4, bidirectional=False)
    bm, sq, sp = o.samples
    nodelim = gpu.Index.from_bwt(5, o.bwt, o.bwt_rev, bm, sq, sp, no_delim=True)
    quni, qnd = uni.upload(sym, off), nodelim.upload(sym, off)
    r = C.c_void_p()
    before = capi.kernel_launch_count()
    assert L.fmb_search_smems(uni.h, quni.h, C.c_uint32(0), C.byref(r)) == -5
    assert L.fmb_search_smems(nodelim.h, qnd.h, C.c_uint32(0), C.byref(r)) == -5
    assert L.fmb_locate_smems(uni.h, smems.h, C.c_uint64(1), C.byref(r)) == -5
    assert L.fmb_locate_smems(index.h, hits.h, C.c_uint64(1), C.byref(r)) == -1
    assert L.fmb_locate(index.h, smems.h, C.byref(r)) == -1
    for kind_wrong in (lambda: hits.smems(), lambda: smems.hits(), lambda: smems.locs(), lambda: smems.locs32(), lambda: smems.smem_locs()):
        with pytest.raises(capi.FmbError) as ex:
            kind_wrong()
        assert ex.value.code == -1
    assert capi.kernel_launch_count() == before
    located = index.locate_smems(smems)
    for kind_wrong in (lambda: located.smems(), lambda: located.locs(), lambda: located.hits()):
        with pytest.raises(capi.FmbError) as ex:
            kind_wrong()
        assert ex.value.code == -1


# ---- scale ----------------------------------------------------------------------------------------------------------------------------
def test_scale_certificate(gpu):
    from fmb200 import capi
    n, nq, L = 64_000_000, 1_000_000, 150
    d_text = capi.synth_text_device(0, 5, n, 11)
    try:
        index = gpu.Index.build_from_device_text(5, d_text, n, sampling_rate=16)
        d_reads = capi.synth_reads_err_device(0, d_text, n, nq, L, 17, 5, 6, True)
        sym = np.zeros(nq * L, dtype=np.uint8)
        capi.copy_to_host(0, sym, d_reads, nq * L)
        capi.device_free(0, d_reads)
    finally:
        capi.device_free(0, d_text)
    off = np.arange(nq + 1, dtype=np.uint64) * np.uint64(L)
    q = index.upload(sym, off)
    r0 = index.search_smems(q, min_len=0)
    all_smems = r0.smems()
    assert certify(index, sym, off, all_smems)
    long_smems = index.search_smems(q, min_len=19).smems()
    assert np.array_equal(long_smems, all_smems[(all_smems["end"] - all_smems["begin"]) >= 19])
    loc = index.locate_smems(r0, max_occ=500).smem_locs()
    assert loc.size >= all_smems.size // 2
    # a located row of an SMEM is where the text holds it
    pick = loc[np.random.default_rng(1).choice(loc.size, 2000, replace=False)]
    got = index.extract(pick["seq"], pick["pos"], pick["pos"] + (pick["end"] - pick["begin"]))
    for p, g in zip(pick, got):
        b = int(off[int(p["qidx"])]) + int(p["begin"])
        assert np.array_equal(g, sym[b:b + g.size])


# ---- C++ -------------------------------------------------------------------------------------------------------------------------------
def test_cpp_bulk_and_delegate_forms(gpu, tmp_path):
    binary = str(tmp_path / "smem_test")
    lib = os.path.join(ROOT, "fmindex-collection_b200")
    subprocess.run(["g++", "-std=c++20", "-O2", "-Wall", "-Wno-comment", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "smem_test.cpp"), "-L", lib, "-lfmb200", "-Wl,-rpath," + lib, "-pthread",
                    "-o", binary], check=True)
    r = subprocess.run([binary], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr
