"""CPU tests (no GPU): pin the C oracle (oracle/fm_oracle.c) against
  (1) the literal expectations of the reference's own test-suite (src/test_fmindex-collection/...), restated here,
  (2) tests/golden/ref_vectors.json = outputs of the reference itself (tests/golden/make_golden.py), and
  (3) the reference library oracle/_ref/libfmref.so when it is present (differential, seeded).
"""
import json
import os

import numpy as np
import pytest

from oracle.pyoracle import Oracle, Ref, sort_hits, sort_locs

HERE = os.path.dirname(os.path.abspath(__file__))


def A(s):
    return np.frombuffer(s.encode(), dtype=np.uint8)


def located(o, hits):
    return sorted((int(r["qidx"]), int(r["seq"]), int(r["pos"])) for r in o.locate(hits))


def flat(queries):
    from fmb200 import synth
    return synth.flatten([np.asarray(q, dtype=np.uint8) for q in queries])


# ---- string/unittest.cpp:52-312 "Hallo Welt": hand-counted rank / exclusive prefix_rank -------------------
def test_string_hallo_welt():
    text = A("Hallo Welt")
    o = Oracle.from_bwt(256, text, None, np.zeros(1, dtype=np.uint64), [], [])
    assert [o.symbol(i) for i in range(10)] == list(text)
    assert o.rank(0, ord("H")) == 0 and o.rank(1, ord("H")) == 1 and o.rank(10, ord("l")) == 3
    assert o.rank(3, ord("l")) == 1 and o.rank(4, ord("l")) == 2 and o.rank(9, ord("l")) == 3
    # prefix_rank is exclusive ("<"): string/unittest.cpp:203,215
    assert o.prefix_rank(1, ord("H")) == 0 and o.prefix_rank(1, ord("W")) == 1
    assert o.prefix_rank(10, ord("a")) == 3          # ' ', 'H', 'W' sort before 'a'
    rs, prs = o.all_ranks_and_prefix_ranks(10)
    assert rs[ord("l")] == 3 and rs[ord("o")] == 1 and prs[ord("l")] == 5 and prs[0] == 0
    for i in range(11):
        rs, prs = o.all_ranks_and_prefix_ranks(i)
        for c in (32, 72, 87, 97, 101, 108, 111, 116):
            assert rs[c] == o.rank(i, c) and prs[c] == o.prefix_rank(i, c)


# ---- fmindex/checkBiFMIndexCursor.cpp:12-103 ---------------------------------------------------------------
def test_cursor_1111222():
    text = np.array([1, 1, 1, 1, 2, 2, 2, 0], dtype=np.uint8)
    o = Oracle.build(text, 5, 1)
    root = [0, 0, o.n, 0]
    assert o.n == 8
    for right in (0, 1):
        for s, (cnt, lb) in {0: (1, 0), 1: (4, 1), 2: (3, 5), 3: (0, 8)}.items():
            c = o.extend(root, s, right)
            assert (c[2], c[1] if right else c[0]) == (cnt, lb)
        allc = o.extend_all(root, right)
        for s in range(5):
            assert np.array_equal(allc[s], o.extend(root, s, right))


# ---- fmindex/checkBiFMIndex.cpp:13-105: locate under three sampling patterns -------------------------------
@pytest.mark.parametrize("pattern", ["full", "even_rows", "odd_rows", "even_text"])
def test_locate_hallo_welt(pattern):
    bwt = np.array([ord(c) if c != "$" else 0 for c in "t$o$ HWalell"], dtype=np.uint8)
    bwt_rev = np.array([ord(c) if c != "$" else 0 for c in "H$Waelllto $"], dtype=np.uint8)
    sa = [10, 11, 5, 0, 6, 1, 7, 2, 3, 8, 4, 9]
    keep = {
        "full": [True] * 12,
        "even_rows": [(i % 2 == 0) or sa[i] == 0 for i in range(12)],
        "odd_rows": [i % 2 == 1 for i in range(12)],
        "even_text": [sa[i] % 2 == 0 for i in range(12)],
    }[pattern]
    bitmap = np.zeros(1, dtype=np.uint64)
    seq, pos = [], []
    for i, k in enumerate(keep):
        if k:
            bitmap[0] |= np.uint64(1) << np.uint64(i)
            seq.append(0)
            pos.append(sa[i])
    o = Oracle.from_bwt(255, bwt, bwt_rev, bitmap, seq, pos)
    for i in range(12):
        s, p, off = o.locate_row(i)
        assert s == 0 and p + off == sa[i]
        step = o.single_locate_step(i)
        if keep[i]:
            assert step == (0, sa[i]) and off == 0
        else:
            assert step is None


# ---- search/checkSearchBacktracking.cpp:12-100: literal BWT of a two-sequence collection -------------------
def test_backtracking_collection_bwt():
    t1 = np.concatenate([A("AAACAAACAAA"), [0]]).astype(np.uint8)
    o = Oracle.build(t1, 255, 1)
    assert [o.symbol(i) for i in range(12)] == [65, 65, 65, 67, 67, 0, 65, 65, 65, 65, 65, 65]
    sym, off = flat([A("A")])
    h = o.search_backtracking(sym, off, 0)
    assert len(h) == 1 and h[0]["lb"] == 1 and h[0]["len"] == 9 and h[0]["e"] == 0
    t2 = np.concatenate([A("AAACAAACAAA"), [0], A("AAABAAABAAA"), [0]]).astype(np.uint8)
    o = Oracle.build(t2, 255, 1)
    expected = list(A("AAAAAABCB")) + [0] + [67, 0] + [65] * 12
    assert [o.symbol(i) for i in range(24)] == expected
    h = o.search_backtracking(sym, off, 0)
    assert len(h) == 1 and h[0]["lb"] == 2 and h[0]["len"] == 18


# ---- search/checkSearches.cpp: one fixture, expected located hits for every algorithm ----------------------
@pytest.fixture(scope="module")
def check_searches():
    text = np.concatenate([A("AAACAAABAAA"), [0], A("AAABAAACAAA"), [0]]).astype(np.uint8)
    return Oracle.build(text, 256, 1)


HAM = [(0, 0, 2), (0, 0, 3), (0, 1, 6), (0, 1, 7), (1, 0, 6), (1, 0, 7), (1, 1, 2), (1, 1, 3)]
PIGEON_OPT_K1 = (np.array([[0, 1], [1, 0]]), np.array([[0, 0], [0, 1]]), np.array([[0, 1], [0, 1]]))


def test_checkSearches_backtracking_and_exact(check_searches):
    o = check_searches
    sym, off = flat([A("CC"), A("BB")])
    assert located(o, o.search_backtracking(sym, off, 1)) == HAM                      # :23-102
    assert located(o, o.search_exact(sym, off)) == []                                 # :104-117


def test_checkSearches_ng26(check_searches):
    from fmb200 import schemes
    o = check_searches
    part = schemes.uniform_partition(2, 2)
    sym, off = flat([A("CD"), A("DB")])
    assert located(o, o.search_ng26(sym, off, PIGEON_OPT_K1, part, True)) == [(0, 0, 3), (0, 1, 7), (1, 0, 7), (1, 1, 3)]   # :1093-1120
    sym, off = flat([A("CC"), A("BB")])
    assert located(o, o.search_ng26(sym, off, PIGEON_OPT_K1, part, False)) == HAM     # :1174-1199
    # :1148-1172 search_n = 3 (clipping of the last cursor, SearchNg26.h:414-421)
    exp_n3 = [(0, 0, 3), (0, 1, 7), (0, 1, 7), (1, 0, 7), (1, 0, 7), (1, 1, 3)]
    assert located(o, o.search_ng26(sym, off, PIGEON_OPT_K1, part, True, max_hits=3)) == exp_n3


def test_checkSearches_facade(check_searches):
    from fmb200 import schemes
    o = check_searches
    sym, off = flat([A("CC"), A("BB")])
    sch, part = schemes.facade_scheme(True, 1, 2)
    exp = [(0, 0, 3), (0, 0, 3), (0, 1, 7), (0, 1, 7), (1, 0, 7), (1, 0, 7), (1, 1, 3), (1, 1, 3)]
    assert located(o, o.search_ng26(sym, off, sch, part, True)) == exp                # :1422-1444
    exp_n3 = [(0, 0, 3), (0, 1, 7), (0, 1, 7), (1, 0, 7), (1, 0, 7), (1, 1, 3)]
    assert located(o, o.search_ng26(sym, off, sch, part, True, max_hits=3)) == exp_n3  # :1446-1466
    sch, part = schemes.facade_scheme(False, 1, 2)
    assert located(o, o.search_ng26(sym, off, sch, part, False)) == HAM               # :1468-1490


# ---- golden vectors produced by the reference itself -------------------------------------------------------
@pytest.fixture(scope="module")
def golden():
    with open(os.path.join(HERE, "golden", "ref_vectors.json")) as f:
        return json.load(f)


def _hits_arr(rows):
    from oracle.pyoracle import HIT_DTYPE
    a = np.zeros(len(rows), dtype=HIT_DTYPE)
    for i, r in enumerate(rows):
        a[i] = tuple(r)
    return a


def _locs_arr(rows):
    from oracle.pyoracle import LOC_DTYPE
    a = np.zeros(len(rows), dtype=LOC_DTYPE)
    for i, r in enumerate(rows):
        a[i] = tuple(r)
    return a


def test_scheme_generators_match_reference(golden):
    from fmb200 import schemes
    g = golden["schemes"]
    for (mn, mx) in ((0, 0), (0, 1), (0, 2), (1, 2)):
        assert [a.astype(int).tolist() for a in schemes.optimum(mn, mx)] == g[f"optimum:{mn}:{mx}"]
    for k in (1, 2, 3):
        for extra in (1, 2, 3):
            assert [a.astype(int).tolist() for a in schemes.h2(k + extra, 0, k)] == g[f"h2-k{extra}:0:{k}"]
        assert [a.astype(int).tolist() for a in schemes.backtracking(1, 0, k)] == g[f"backtracking:0:{k}"]
    assert [a.astype(int).tolist() for a in schemes.h2(4, 1, 2)] == g["h2-k2:1:2"]


@pytest.mark.parametrize("case", [0, 1, 2])
def test_oracle_matches_reference_vectors(golden, case):
    from fmb200 import schemes, synth
    c = golden["cases"][case]
    text = np.array(c["text"], dtype=np.uint8)
    assert np.array_equal(text, synth.multi_text(c["lengths"], 5, c["seed"]))          # generator is stable
    o = Oracle.build(text, 5, c["rate"])
    n = o.n
    assert [o.symbol(i, 0) for i in range(n)] == c["bwt"]                              # suffix sort + BWT (utils.h:97-163)
    assert [o.symbol(i, 1) for i in range(n)] == c["bwt_rev"]                          # BiFMIndex.h:82-91
    assert [int(x) for x in o.C] == c["C"]
    assert [list(o.locate_row(i)) for i in range(n)] == c["locate_all"]                # sampling + LF walk
    for s in c["string"]:
        assert [o.rank(s["row"], k, s["dir"]) for k in range(5)] == s["rank"]
        assert [o.prefix_rank(s["row"], k, s["dir"]) for k in range(6)] == s["prefix_rank"]
    sym, off = synth.flatten(np.array(c["queries"], dtype=np.uint8))
    S = c["searches"]
    h = o.search_exact(sym, off)
    assert np.array_equal(sort_hits(h), _hits_arr(S["exact"]["hits"]))
    assert np.array_equal(sort_locs(o.locate(h)), _locs_arr(S["exact"]["locs"]))
    for k in (1, 2):
        for edit in (False, True):
            tag = "edit" if edit else "ham"
            sch = schemes.optimum(0, k)
            part = schemes.uniform_partition(sch[0].shape[1], c["L"])
            h = o.search_ng26(sym, off, sch, part, edit)
            assert np.array_equal(sort_hits(h), _hits_arr(S[f"ng26_optimum_k{k}_{tag}"]["hits"])), (k, edit)
            assert np.array_equal(sort_locs(o.locate(h)), _locs_arr(S[f"ng26_optimum_k{k}_{tag}"]["locs"]))
            sch, part = schemes.facade_scheme(edit, k, c["L"])
            h = o.search_ng26(sym, off, sch, part, edit)
            assert np.array_equal(sort_hits(h), _hits_arr(S[f"facade_k{k}_{tag}"]["hits"])), ("facade", k, edit)
    ssym, soff = synth.flatten(np.array(c["short_queries"], dtype=np.uint8))
    for k in (0, 1, 2):
        assert np.array_equal(sort_hits(o.search_backtracking(ssym, soff, k)), _hits_arr(S[f"backtracking_k{k}"]["hits"]))


def test_hit_limited_searches_match_reference_output_in_order(golden):
    """search_ng26::search(..., n) (SearchNg26.h:408-433): the reference's delegate calls, in the reference's order, recorded by
    tests/golden/make_golden.py -- random texts and a repetitive collection (wide nodes, cursors with many rows that get clipped)"""
    from fmb200 import schemes, synth
    checked = 0
    for c in list(golden["cases"]) + [golden["hit_limit_case"]]:
        o = Oracle.build(np.array(c["text"], dtype=np.uint8), 5, c["rate"])
        sym, off = synth.flatten(np.array(c["queries"], dtype=np.uint8))
        for key, val in c["searches"].items():
            if "hits_in_order" not in val:
                continue
            _, _, kk, tag, nn = key.split("_")                       # ng26_optimum_k1_edit_n3
            sch = schemes.optimum(0, int(kk[1:]))
            part = schemes.uniform_partition(sch[0].shape[1], c["L"])
            got = o.search_ng26(sym, off, sch, part, tag == "edit", max_hits=int(nn[1:]))
            assert np.array_equal(got, _hits_arr(val["hits_in_order"])), (c["name"], key)
            checked += len(got)
    assert checked > 2000


# ---- live differential against the reference library, when it was built ------------------------------------
@pytest.mark.skipif(not Ref.available(), reason="oracle/_ref/libfmref.so not built (needs /root/reference)")
@pytest.mark.parametrize("seed", [1, 2])
def test_oracle_vs_reference_library(seed):
    from fmb200 import schemes, synth
    text = synth.multi_text([2500, 1200, 33], 5, 50 + seed)
    o = Oracle.build(text, 5, 5)
    r = Ref.build(text, 5, 5)
    assert all(o.symbol(i) == r.symbol(i) and o.symbol(i, 1) == r.symbol(i, 1) for i in range(o.n))
    assert all(o.locate_row(i) == r.locate_row(i) for i in range(0, o.n, 7))
    reads, _ = synth.reads_from_text(text[:2500], 120, 32, seed)
    reads = synth.plant_errors(reads, 5, seed, True, seed)
    sym, off = synth.flatten(reads)
    for k in (1, 2):
        for edit in (False, True):
            sch = schemes.optimum(0, k)
            part = schemes.uniform_partition(sch[0].shape[1], 32)
            a, b = sort_hits(o.search_ng26(sym, off, sch, part, edit)), sort_hits(r.search_ng26(sym, off, sch, part, edit))
            assert np.array_equal(a, b)
            assert np.array_equal(sort_locs(o.locate(a)), sort_locs(r.locate(b)))
    # multi-threaded sharding of the reference arm gives the same multiset
    sch = schemes.optimum(0, 1)
    part = schemes.uniform_partition(2, 32)
    assert np.array_equal(sort_hits(r.search_ng26(sym, off, sch, part, True, threads=3)), sort_hits(r.search_ng26(sym, off, sch, part, True)))


# ---- discovery-order keys (test aid for the device's hit-limited search) -----------------------------------
@pytest.mark.parametrize("kind", ["random", "repeats", "protein"])
def test_discovery_order_keys_ascend_in_report_order(kind):
    """The device enumerates a search tree in its own order and sorts the hits by a sparse key afterwards; the key (defined in
    fm_oracle.c, ng26_key_edge) must therefore ascend strictly in the order the reference's depth-first search reports hits
    (SearchNg26.h:170-218 wide nodes, :286-363 single-row nodes; searches in scheme order :385-390)."""
    from fmb200 import schemes, synth
    rng = np.random.default_rng(11)
    if kind == "random":
        sigma, L = 5, 24
        text = synth.multi_text([1500, 700], sigma, 5)
    elif kind == "repeats":
        sigma, L = 5, 20
        unit = rng.integers(1, 5, 40).astype(np.uint8)
        chunks = []
        for _ in range(40):
            u = unit.copy()
            u[rng.integers(0, 40, 2)] = rng.integers(1, 5, 2)
            chunks.append(u)
        text = np.concatenate(chunks + [np.zeros(1, np.uint8)])
    else:
        sigma, L = 21, 12
        text = synth.multi_text([900, 300], sigma, 9)
    o = Oracle.build(text, sigma, 4)
    body = text[: 700 if kind != "repeats" else len(text) - 1]
    reads, _ = synth.reads_from_text(body, 60, L, 3)
    reads = synth.plant_errors(reads, sigma, 2, True, 4)
    sym, off = synth.flatten(reads)
    total = 0
    for k in (1, 2, 3):
        for edit in (False, True):
            for sch in (schemes.optimum(0, k) if k < 3 else schemes.h2(k + 2, 0, k), schemes.h2(k + 1, 0, k), schemes.backtracking(k + 1, 0, k)):
                if not edit:
                    sch = schemes.limit_to_hamming(sch)
                part = schemes.uniform_partition(sch[0].shape[1], L)
                hits, keys = o.search_ng26_keys(sym, off, sch, part, edit)
                assert np.array_equal(hits, o.search_ng26(sym, off, sch, part, edit))
                same_q = hits["qidx"][1:] == hits["qidx"][:-1]
                assert np.all(keys[1:][same_q] > keys[:-1][same_q]), (kind, k, edit)
                total += hits.size
    assert total > 500


# ---- search_pseudo (search/SearchPseudo.h): golden literals + live differential ----------------------------
def test_checkSearches_pseudo(check_searches):
    """search/checkSearches.cpp:143-176 (edit distance, 'all search') and :215-241 (Hamming) with expand(pigeon_opt(0,1), 2)"""
    from fmb200 import schemes
    o = check_searches
    sym, off = flat([A("CC"), A("BB")])
    expanded = schemes.expand(PIGEON_OPT_K1, [1, 1])
    exp_edit = [(0, 0, 2), (0, 0, 3), (0, 0, 3), (0, 0, 3), (0, 1, 6), (0, 1, 7), (0, 1, 7), (0, 1, 7),
                (1, 0, 6), (1, 0, 7), (1, 0, 7), (1, 0, 7), (1, 1, 2), (1, 1, 3), (1, 1, 3), (1, 1, 3)]
    assert located(o, o.search_pseudo(sym, off, expanded, True)) == exp_edit
    assert located(o, o.search_pseudo(sym, off, expanded, False)) == HAM


def _pseudo_inputs():
    from fmb200 import synth
    text = synth.multi_text([1800, 600], 5, 61)
    L = 18
    reads, _ = synth.reads_from_text(text[:1800], 60, L, 5)
    reads = synth.plant_errors(reads, 5, 1, True, 6)
    return text, L, *synth.flatten(reads)


def _pseudo_schemes(k):
    from fmb200 import schemes
    return schemes.optimum(0, k), schemes.h2(k + 2, 0, k), schemes.backtracking(k + 1, 0, k)


@pytest.mark.skipif(not Ref.available(), reason="oracle/_ref/libfmref.so not built (needs /root/reference)")
def test_pseudo_oracle_vs_reference_library():
    from fmb200 import schemes
    text, L, sym, off = _pseudo_inputs()
    o = Oracle.build(text, 5, 4)
    r = Ref.build(text, 5, 4)
    total = 0
    for k in (1, 2):
        for sch in _pseudo_schemes(k):
            expanded = schemes.expand(sch, schemes.uniform_partition(sch[0].shape[1], L))
            for edit in (False, True):
                a, b = sort_hits(o.search_pseudo(sym, off, expanded, edit)), sort_hits(r.search_pseudo(sym, off, expanded, edit))
                assert np.array_equal(a, b), (k, edit)
                total += len(a)
    assert total > 1000


def test_pseudo_hamming_equals_ng26():
    """Hamming: the per-symbol search equals the per-part search of search_ng26 (the argument behind the device's fold)"""
    from fmb200 import schemes
    text, L, sym, off = _pseudo_inputs()
    o = Oracle.build(text, 5, 4)
    for k in (1, 2):
        for sch in _pseudo_schemes(k):
            ham = schemes.limit_to_hamming(sch)
            part = schemes.uniform_partition(sch[0].shape[1], L)
            assert np.array_equal(sort_hits(o.search_pseudo(sym, off, schemes.expand(ham, part), False)), sort_hits(o.search_ng26(sym, off, ham, part, False)))


def test_pseudo_hamming_matches_reference_vectors(golden):
    """search_pseudo with Hamming distance on the expanded scheme reports exactly the hits of the reference's own search_ng26 and
    search facade on the unexpanded one (tests/golden/ref_vectors.json): anchors the oracle's search_pseudo, which the device's
    pseudo search is checked against, on outputs of the reference"""
    from fmb200 import schemes, synth
    total = 0
    for c in golden["cases"]:
        o = Oracle.build(np.array(c["text"], dtype=np.uint8), 5, c["rate"])
        sym, off = synth.flatten(np.array(c["queries"], dtype=np.uint8))
        for k in (1, 2):
            sch = schemes.optimum(0, k)
            for key, (s, part) in ((f"ng26_optimum_k{k}_ham", (sch, schemes.uniform_partition(sch[0].shape[1], c["L"]))),
                                   (f"facade_k{k}_ham", schemes.facade_scheme(False, k, c["L"]))):
                got = sort_hits(o.search_pseudo(sym, off, schemes.expand(s, part), False))
                assert np.array_equal(got, _hits_arr(c["searches"][key]["hits"])), (c["name"], key)
                total += len(got)
    assert total > 250
