"""Text extraction on the GPU (fmb_extract, fmb_index_reconstruct_text, fmb_index_sequence_lengths; reconstructText utils.h:672): the
text read back from an index equals the text the index was built from, on every table configuration and sampling the library accepts,
and the refusals launch nothing."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

from helpers import Oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FMB_TABLE_JUMP, FMB_TABLE_JUMP4, FMB_TABLE_JUMP32, FMB_TABLE_ANCHORS = 4, 128, 256, 512


def collection(sigma, count, seed, min_len=1, max_len=200):
    rng = np.random.default_rng(seed)
    seqs = [rng.integers(1, sigma, size=int(rng.integers(min_len, max_len + 1)), dtype=np.uint8) for _ in range(count)]
    text = np.concatenate([np.append(s, np.uint8(0)) for s in seqs]).astype(np.uint8)
    return seqs, text


def random_ranges(seqs, count, seed):
    """random ranges plus the edge cases: empty, single symbols, whole sequences, ranges ending at a sequence end and starting at 0"""
    rng = np.random.default_rng(seed)
    lens = np.array([len(s) for s in seqs], dtype=np.int64)
    seq = rng.integers(0, len(seqs), size=count)
    b = (rng.random(count) * (lens[seq] + 1)).astype(np.int64)
    e = b + (rng.random(count) * (lens[seq] - b + 1)).astype(np.int64)
    k = np.arange(min(len(seqs), 50))
    extra = [
        (k, np.zeros_like(k), np.zeros_like(k)),                      # empty at 0
        (k, lens[k], lens[k]),                                        # empty at the end
        (k, np.zeros_like(k), np.minimum(lens[k], 1)),                # first symbol
        (k, np.maximum(lens[k] - 1, 0), lens[k]),                     # last symbol
        (k, np.zeros_like(k), lens[k]),                               # whole sequence
        (k, lens[k] // 2, lens[k]),                                   # ending at the sequence end
        (k, np.zeros_like(k), lens[k] // 2),                          # starting at 0
    ]
    for s, bb, ee in extra:
        seq, b, e = np.concatenate([seq, s]), np.concatenate([b, bb]), np.concatenate([e, ee])
    return seq.astype(np.uint64), b.astype(np.uint64), e.astype(np.uint64)


def check_ranges(index, seqs, seq, b, e):
    got, st = index.extract(seq, b, e, with_stats=True)
    for i in range(len(seq)):
        want = seqs[int(seq[i])][int(b[i]):int(e[i])]
        assert np.array_equal(got[i], want), (i, int(seq[i]), int(b[i]), int(e[i]))
    return st


def check_index(index, seqs, text, seed=5, count=3000):
    assert np.array_equal(index.sequence_lengths(), np.array([len(s) for s in seqs], dtype=np.uint64))
    assert np.array_equal(index.reconstruct_text(), text)
    return check_ranges(index, seqs, *random_ranges(seqs, count, seed))


def row_sampled_index(gpu, text, sigma, bidirectional=True, every=2):
    """fmb_index_create from BWT + samples with row-space sampling ("every 2nd row", the reference's checkBiFMIndex.cpp): the sample
    of a row is (seq, pos) of its suffix, so position 0 of a sequence is not always sampled"""
    o = Oracle.build(text, sigma, 1, bidirectional)
    sa = np.asarray(o.sa, dtype=np.int64)
    n = sa.size
    delims = np.flatnonzero(text == 0)
    rows = np.arange(0, n, every)
    p = sa[rows]
    seq = np.searchsorted(delims, p, side="left")
    pos = p - np.where(seq > 0, delims[np.maximum(seq - 1, 0)] + 1, 0)
    bits = np.zeros(n, dtype=bool)
    bits[rows] = True
    packed = np.packbits(bits, bitorder="little")
    packed = np.concatenate([packed, np.zeros((-packed.size) % 8, dtype=np.uint8)])
    bm = packed.view("<u8")
    return gpu.Index.from_bwt(sigma, o.bwt, o.bwt_rev if bidirectional else None, bm, seq.astype(np.uint32), pos.astype(np.uint32)), o


@pytest.mark.parametrize("sigma", [5, 21])
def test_round_trip_short_sequences(gpu, tmp_path, sigma):
    seqs, text = collection(sigma, 300, 11 + sigma)
    index = gpu.Index.build(sigma, text, sampling_rate=4)
    st = check_index(index, seqs, text)
    assert st.line_requests > 0                          # sigma = 5: LF^16 / LF^4 jumps; sigma = 21: byte LF^4 jumps
    assert index.info.tables & FMB_TABLE_ANCHORS
    path = str(tmp_path / "ix.fmb")
    index.save(path)
    loaded = gpu.Index.load(path)
    assert not loaded.info.tables & FMB_TABLE_ANCHORS    # built on first use, not stored
    check_index(loaded, seqs, text, seed=6)


@pytest.fixture(scope="module")
def mbp(gpu):
    seqs, text = collection(5, 40, 3, min_len=1, max_len=50_000)
    return seqs, text


def test_one_mbp_every_table(gpu, mbp):
    seqs, text = mbp
    index = gpu.Index.build(5, text, sampling_rate=16)
    t = index.info.tables
    assert t & FMB_TABLE_JUMP and t & FMB_TABLE_JUMP4 and t & FMB_TABLE_JUMP32
    before = index.info.device_bytes
    st = check_index(index, seqs, text, count=20000)
    assert index.info.device_bytes > before
    symbols = len(text) - len(seqs)
    st_whole = check_ranges(index, seqs, np.arange(len(seqs), dtype=np.uint64), np.zeros(len(seqs), dtype=np.uint64),
                            np.array([len(s) for s in seqs], dtype=np.uint64))
    # whole sequences at rate 16: about one LF^16 request per 16 symbols, few single steps
    assert st_whole.line_requests <= symbols // 16 + 4 * len(seqs) + 16
    assert st_whole.lf_steps < symbols // 16
    assert st.line_requests > 0


@pytest.mark.parametrize("knob", ["FMB_NO_JUMP", "FMB_NO_JUMP32", "FMB_NO_JUMP4"])
def test_one_mbp_without_tables(gpu, mbp, monkeypatch, knob):
    seqs, text = mbp
    monkeypatch.setenv(knob, "1")                        # read when the index is built
    index = gpu.Index.build(5, text, sampling_rate=16)
    monkeypatch.delenv(knob)
    t = index.info.tables
    st = check_index(index, seqs, text, count=5000)
    if knob == "FMB_NO_JUMP":
        assert not t & (FMB_TABLE_JUMP | FMB_TABLE_JUMP4)
        assert st.line_requests == 0 and st.lf_steps > 0
    elif knob == "FMB_NO_JUMP32":
        assert t & FMB_TABLE_JUMP and not t & FMB_TABLE_JUMP32
        assert st.line_requests > 0
    else:
        assert t & FMB_TABLE_JUMP and not t & FMB_TABLE_JUMP4
        assert st.line_requests > 0 and st.lf_steps > 0


@pytest.mark.parametrize("sigma", [5, 21])
def test_row_sampled_index(gpu, sigma):
    seqs, text = collection(sigma, 300, 21 + sigma)
    index, o = row_sampled_index(gpu, text, sigma)
    # position 0 of some sequence is not sampled, and some short sequences hold no sample at all
    check_index(index, seqs, text)


def test_unidirectional_index(gpu):
    seqs, text = collection(5, 200, 31)
    index = gpu.Index.build(5, text, sampling_rate=8, bidirectional=False)
    check_index(index, seqs, text)
    index, _ = row_sampled_index(gpu, text, 5, bidirectional=False, every=3)
    check_index(index, seqs, text, seed=9)


def _edit_within(query, ref, e):
    """min over m of the edit distance of query and ref[:m] is <= e (ref starts where the hit starts)"""
    q = np.asarray(query, dtype=np.int64)
    r = np.asarray(ref, dtype=np.int64)
    prev = np.arange(r.size + 1)                          # row 0: distance of "" to ref[:m]
    for i in range(1, q.size + 1):
        cur = np.empty_like(prev)
        cur[0] = i
        sub = prev[:-1] + (r != q[i - 1])
        dele = prev[1:] + 1
        best = np.minimum(sub, dele)
        for m in range(1, r.size + 1):                    # insertions along the row
            cur[m] = min(best[m - 1], cur[m - 1] + 1)
        prev = cur
    return int(prev.min()) <= e


def test_hits_match_extracted_reference(gpu):
    from fmb200 import schemes
    seqs, text = collection(5, 60, 41, min_len=200, max_len=2000)
    index = gpu.Index.build(5, text, sampling_rate=16)
    rng = np.random.default_rng(4)
    L, nq = 40, 300
    reads = []
    for _ in range(nq):
        s = seqs[int(rng.integers(len(seqs)))]
        p = int(rng.integers(0, len(s) - L))
        r = list(s[p:p + L])
        for _ in range(int(rng.integers(0, 3))):
            k = int(rng.integers(L))
            r[k] = 1 + (r[k] % 4)
        reads.append(r)
    sym = np.array(reads, dtype=np.uint8).reshape(-1)
    off = np.arange(nq + 1, dtype=np.uint64) * np.uint64(L)
    locs, _ = index.search_and_locate(sym, off, scheme=schemes.optimum(0, 2), partition=schemes.uniform_partition(4, L), edit=True,
                                      capacity=nq * 1000)
    assert len(locs) >= nq
    lens = index.sequence_lengths()
    pick = locs[np.random.default_rng(5).choice(len(locs), min(400, len(locs)), replace=False)]
    seq = pick["seq"].astype(np.uint64)
    b = pick["pos"].astype(np.uint64)
    e = np.minimum(b + np.uint64(L + 2), lens[seq])
    got = index.extract(seq, b, e)
    for h, ref in zip(pick, got):
        q = reads[int(h["qidx"])]
        assert np.array_equal(ref, seqs[int(h["seq"])][int(h["pos"]):int(h["pos"]) + len(ref)])
        assert _edit_within(q, ref, int(h["e"])), (int(h["qidx"]), int(h["e"]))


def test_refusals_launch_nothing(gpu):
    from fmb200 import capi
    L = capi.lib()
    seqs, text = collection(5, 20, 51)
    index = gpu.Index.build(5, text, sampling_rate=4)
    lens = index.sequence_lengths()                       # builds the sequence layout
    index.extract(0, 0, 1)                                # and the anchor table
    n_seq = len(seqs)

    def call(seq, b, e, capacity):
        seq, b, e = (np.array(x, dtype=np.uint64) for x in (seq, b, e))
        out = np.zeros(max(capacity, 1), dtype=np.uint8)
        off = np.zeros(seq.size + 1, dtype=np.uint64)
        before = capi.kernel_launch_count()
        rc = L.fmb_extract(index.h, capi._ptr(seq), capi._ptr(b), capi._ptr(e), C.c_uint64(seq.size), capi._ptr(out),
                           C.c_uint64(capacity), capi._ptr(off), None)
        assert capi.kernel_launch_count() == before
        return rc, off

    assert call([n_seq], [0], [0], 100)[0] == -1                               # seq out of range
    assert call([0], [2], [1], 100)[0] == -1                                   # begin > end
    assert call([0], [0], [int(lens[0]) + 1], 100)[0] == -1                    # end > length
    rc, off = call([0, 1], [0, 0], [lens[0], lens[1]], int(lens[0]))          # capacity short by lens[1]
    assert rc == -1 and int(off[-1]) == int(lens[0] + lens[1])
    out = np.zeros(len(text) - 1, dtype=np.uint8)
    before = capi.kernel_launch_count()
    assert L.fmb_index_reconstruct_text(index.h, capi._ptr(out), C.c_uint64(out.size)) == -1
    assert capi.kernel_launch_count() == before

    o = Oracle.build(text, 5, 4, False)
    bm, sq, sp = o.samples
    nodelim = gpu.Index.from_bwt(5, o.bwt, None, bm, sq, sp, no_delim=True)
    before = capi.kernel_launch_count()
    for f in (nodelim.sequence_count, nodelim.sequence_lengths, nodelim.reconstruct_text, lambda: nodelim.extract(0, 0, 1)):
        with pytest.raises(capi.FmbError) as ex:
            f()
        assert ex.value.code == -5
    assert capi.kernel_launch_count() == before


def test_concurrent_first_use_builds_once(gpu, mbp):
    seqs, text = mbp
    index = gpu.Index.build(5, text, sampling_rate=16)
    before = index.info.device_bytes
    seq, b, e = random_ranges(seqs, 2000, 61)
    errors, barrier = [], threading.Barrier(2)

    def work():
        try:
            barrier.wait()
            check_ranges(index, seqs, seq, b, e)
        except Exception as ex:                           # noqa: BLE001 -- reported below
            errors.append(ex)

    threads = [threading.Thread(target=work) for _ in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    info = index.info
    assert info.tables & FMB_TABLE_ANCHORS
    assert info.device_bytes - before == 8 * (info.n_samples + info.n_delims)   # one table
    check_ranges(index, seqs, seq, b, e)
    assert index.info.device_bytes == info.device_bytes


def test_image_budget_refuses_anchor_table(gpu):
    from fmb200 import capi
    seqs, text = collection(5, 50, 71)
    index = gpu.Index.build(5, text, sampling_rate=4)
    try:
        capi.set_image_budget(index.info.device_bytes + 1)
        with pytest.raises(capi.FmbError) as ex:
            index.reconstruct_text()
        assert ex.value.code == -4
    finally:
        capi.set_image_budget(0)
    assert not index.info.tables & FMB_TABLE_ANCHORS
    check_index(index, seqs, text)                       # still usable


def test_scale_64_mbp(gpu):
    from fmb200 import capi
    n = 64_000_000
    d_text = capi.synth_text_device(0, 5, n, 11)
    try:
        index = gpu.Index.build_from_device_text(5, d_text, n, sampling_rate=16, bidirectional=True, device=0)
        text = np.zeros(n, dtype=np.uint8)
        capi.copy_to_host(0, text, d_text, n)
    finally:
        capi.device_free(0, d_text)
    assert np.array_equal(index.reconstruct_text(), text)
    rng = np.random.default_rng(8)
    b = rng.integers(0, n - 1 - 150, size=100_000).astype(np.uint64)
    e = b + rng.integers(0, 151, size=b.size).astype(np.uint64)
    got = index.extract(np.zeros(b.size, dtype=np.uint64), b, e)
    for i in range(b.size):
        assert np.array_equal(got[i], text[int(b[i]):int(e[i])]), i


def test_cpp_reconstruct_and_partitioned_extract(gpu, tmp_path):
    binary = str(tmp_path / "extract_test")
    lib = os.path.join(ROOT, "fmindex-collection_b200")
    subprocess.run(["g++", "-std=c++20", "-O2", "-Wall", "-Wno-comment", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "extract_test.cpp"), "-L", lib, "-lfmb200", "-Wl,-rpath," + lib, "-pthread",
                    "-o", binary], check=True)
    r = subprocess.run([binary], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr
