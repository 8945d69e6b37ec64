"""C++ host side (include/fmb200/*.hpp): the reference's search API over the C-ABI.

CPU part: the headers compile as C++20 and the test binary fails loudly without a device (no CPU fallback).
GPU part: tests/cpp/shim_test (shim vs the oracle) and tests/cpp/dropin_test (the reference's own fmc:: calls vs the
fmb200:: calls on fmb200::attach(index), same delegate code; prebuilt here because it needs /root/reference)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "_bin")


def _build():
    import fmb200  # noqa: F401  builds libfmb200.so if needed
    from fmb200 import build as b
    b.build()
    subprocess.run(["bash", os.path.join(ROOT, "tests", "cpp", "build.sh")], check=True, capture_output=True)


def _binary(name):
    path = os.path.join(BIN, name)
    if not os.path.exists(path) and name == "shim_test":
        _build()
    return path


def test_headers_compile_standalone(tmp_path):
    src = tmp_path / "t.cpp"
    src.write_text('#include "fmb200/fmb200.hpp"\nint main() { return fmb200::search_scheme::generator::optimum(0, 2).size() == 3 ? 0 : 1; }\n')
    subprocess.run(["g++", "-std=c++20", "-fsyntax-only", "-Wall", "-Wno-comment", "-I", os.path.join(ROOT, "include"), str(src)], check=True)


def test_scheme_generators_match_python_tables(tmp_path):
    """search_scheme.hpp (C++) against schemes.py, which is pinned to the reference's generators by tests/golden"""
    from fmb200 import schemes
    src = tmp_path / "g.cpp"
    src.write_text(r'''
#include <cstdio>
#include "fmb200/search_scheme.hpp"
namespace ss = fmb200::search_scheme;
static void dump(const char* name, ss::Scheme const& s) {
    std::printf("%s", name);
    for (auto const& x : s) { std::printf(" |"); for (auto v : x.pi) std::printf(" %zu", v); std::printf(" ;"); for (auto v : x.l) std::printf(" %zu", v); std::printf(" ;"); for (auto v : x.u) std::printf(" %zu", v); }
    std::printf("\n");
}
int main() {
    for (size_t k = 0; k <= 3; ++k) for (size_t n = k + 1; n <= k + 3; ++n) { char b[64]; std::snprintf(b, 64, "h2_%zu_%zu", n, k); dump(b, ss::generator::h2(n, 0, k)); std::snprintf(b, 64, "h2h_%zu_%zu", n, k); dump(b, ss::limitToHamming(ss::generator::h2(n, 0, k))); }
    dump("opt_0_1", ss::generator::optimum(0, 1)); dump("opt_0_2", ss::generator::optimum(0, 2)); dump("opt_1_2", ss::generator::optimum(1, 2));
    dump("bt_4_1_2", ss::generator::backtracking(4, 1, 2));
}
''')
    exe = tmp_path / "g"
    subprocess.run(["g++", "-std=c++20", "-O1", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout

    def fmt(name, sch):
        pi, l, u = sch
        parts = [" |" + "".join(f" {v}" for v in pi[s]) + " ;" + "".join(f" {v}" for v in l[s]) + " ;" + "".join(f" {v}" for v in u[s]) for s in range(pi.shape[0])]
        return name + "".join(parts)

    exp = []
    for k in range(4):
        for n in range(k + 1, k + 4):
            exp.append(fmt(f"h2_{n}_{k}", schemes.h2(n, 0, k)))
            exp.append(fmt(f"h2h_{n}_{k}", schemes.limit_to_hamming(schemes.h2(n, 0, k))))
    exp += [fmt("opt_0_1", schemes.optimum(0, 1)), fmt("opt_0_2", schemes.optimum(0, 2)), fmt("opt_1_2", schemes.optimum(1, 2)),
            fmt("bt_4_1_2", schemes.backtracking(4, 1, 2))]
    assert out.strip().splitlines() == exp


def test_shim_binary_fails_loudly_without_device():
    # the devices are hidden from the binary, so that the check also runs where a GPU is present
    r = subprocess.run([_binary("shim_test")], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True)
    assert r.returncode == 2 and "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_shim_against_oracle(gpu):
    r = subprocess.run([_binary("shim_test")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "0 failed" in r.stdout


@pytest.mark.gpu
def test_dropin_against_reference_headers(gpu):
    path = _binary("dropin_test")
    if not os.path.exists(path):
        pytest.skip("tests/cpp/_bin/dropin_test is prebuilt where /root/reference exists (tests/cpp/build.sh)")
    r = subprocess.run([path], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "0 failed" in r.stdout


def test_fasta_front_end(tmp_path):
    """include/fmb200/io.hpp: loadQueries / reverse-complement doubling / result writer (example/utils.h:26-105, main.cpp:260-266)"""
    fa = tmp_path / "reads.fa"
    fa.write_text(">r0 first\nACGT\nTTA\n> r1\nacgtn$\n>r2\n\n>r3\nGGC")          # multi-line record, lower case, empty record, no final newline
    src = tmp_path / "io.cpp"
    src.write_text(r'''
#include <cstdio>
#include "fmb200/fmb200.hpp"
#include "fmb200/io.hpp"
int main(int argc, char** argv) {
    auto [q, info] = fmb200::io::loadQueries<6>(argv[1], true, false);
    for (size_t i = 0; i < q.size(); ++i) {
        std::printf("%s|%d|", info[i].name.c_str(), int(info[i].reverse));
        for (auto c : q[i]) std::printf("%d", int(c));
        std::printf("\n");
    }
    auto [q5, i5] = fmb200::io::loadQueries<5>(argv[1], false, true);               // N -> 1 for Sigma == 5
    for (auto c : q5[1]) std::printf("%d", int(c));
    std::printf("\n");
    bool threw = false;
    try { fmb200::io::loadQueries<5>(argv[1], false, false); } catch (std::runtime_error const&) { threw = true; }
    std::printf("threw=%d missing=%zu\n", int(threw), std::get<0>(fmb200::io::loadQueries<5>("/nonexistent.fa", true, true)).size());
    // packing reader: the same batch as 2-bit words + exception list, equal to what fmb_pack_symbols makes of the flattened bytes
    {
        auto [pq, pinfo] = fmb200::io::loadQueriesPacked<6>(argv[1], true, false);
        bool same = pq.size() == q.size() && pinfo == info;
        auto flat = fmb200::flatten(q);
        same = same && pq.offsets == flat.offsets && pq.symbols() == flat.symbols.size();
        for (size_t i = 0; same && i < flat.symbols.size(); ++i) same = pq.symbol(i) == flat.symbols[i];
        std::vector<uint32_t> words((flat.symbols.size() + 15) / 16 + 1, 0);
        std::vector<uint64_t> ep(flat.symbols.size());
        std::vector<uint8_t> es(flat.symbols.size());
        uint64_t ne = fmb_pack_symbols(flat.symbols.data(), 0, flat.symbols.size(), 5, words.data(), ep.data(), es.data(), ep.size());
        ep.resize(ne); es.resize(ne);
        uint32_t const* w = pq.data();
        same = same && ep == pq.exc_pos && es == pq.exc_sym && pq.words.size() == words.size();
        for (size_t i = 0; same && i < words.size(); ++i) same = w[i] == words[i];
        std::printf("packed=%d exceptions=%zu\n", int(same), pq.exc_pos.size());
    }
    std::vector<std::tuple<size_t, size_t, size_t, size_t>> res{{3, 0, 17, 1}, {4, 1, 2, 0}};
    fmb200::io::saveResults(argv[2], res);
    std::vector<fmb_loc32> res2{{7, 1, 99, 2}};
    fmb200::io::saveResults(std::string(argv[2]) + "2", res2);
}
''')
    exe = tmp_path / "io"
    lib = os.path.join(ROOT, "fmindex-collection_b200")
    import fmb200  # noqa: F401
    from fmb200 import build as b
    b.build()
    subprocess.run(["g++", "-std=c++20", "-O1", "-Wall", "-Wno-comment", "-I", os.path.join(ROOT, "include"), str(src), "-L", lib, "-lfmb200",
                    f"-Wl,-rpath,{lib}", "-o", str(exe)], check=True)
    out = subprocess.run([str(exe), str(fa), str(tmp_path / "out.txt")], check=True, capture_output=True, text=True).stdout.splitlines()
    assert out == ["r0 first|0|1234441", "r0 first|1|4111234", "r1|0|123450", "r1|1|051234", "r2|0|", "r2|1|", "r3|0|332", "r3|1|322",
                   "123410", "threw=1 missing=0", "packed=1 exceptions=4"]
    assert (tmp_path / "out.txt").read_text() == "3 0 17\n4 1 2\n"
    assert (tmp_path / "out.txt2").read_text() == "7 1 99\n"


def test_fold_of_expanded_reference_schemes(tmp_path):
    """search_pseudo's fold() of an expanded scheme re-expands to exactly the same per-symbol scheme -- i.e. the part form handed to
    the device describes the same search -- for the tables of the reference's generators stored in tests/golden/ref_vectors.json
    and many lengths (CPU only: no device call)"""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "ref_vectors.json")) as f:
        tables = {k: v for k, v in json.load(f)["schemes"].items() if k.split(":")[1] == "0" and v[0]}

    def lst(v):
        return "{" + ",".join(str(x) for x in v) + "}"
    literal = ",\n".join("{" + ",".join("{%s,%s,%s}" % (lst(pi), lst(l), lst(u)) for pi, l, u in zip(*t)) + "}" for t in tables.values())
    src = tmp_path / "f.cpp"
    src.write_text(r'''
#include <algorithm>
#include <cstdio>
#include "fmb200/fmb200.hpp"
namespace ms = fmb200::search_scheme;
int main() {
    std::vector<ms::Scheme> schemes = {
''' + literal + r'''
    };
    int checks = 0, bad = 0;
    for (auto const& mine : schemes) {
        for (size_t L : {mine[0].pi.size(), mine[0].pi.size() + 1, size_t{7}, size_t{20}, size_t{50}, size_t{151}}) {
            if (L < mine[0].pi.size()) continue;
            auto e_mine = ms::expand(mine, L);
            if (e_mine.empty()) continue;
            // fold back into parts and expand again with the folded partition: must reproduce pi and u exactly, and a lower bound
            // sequence that accepts exactly the same (position, errors) pairs: max over the prefix is what counts (e never decreases)
            auto [folded, partition] = fmb200::search_pseudo::detail_pseudo::fold(e_mine);
            auto again = ms::expand(folded, partition);
            ++checks;
            bool ok = again.size() == e_mine.size() && partition.size() <= 16;
            for (size_t i = 0; ok && i < again.size(); ++i) {
                // the first part may be walked in either direction (search_ng26 and the device always walk it to the right): same
                // symbols, same bounds -- compare it as a set
                auto first = [&](ms::Search x) { std::sort(x.pi.begin(), x.pi.begin() + partition[folded[i].pi[0]]); return x.pi; };
                ok = first(again[i]) == first(e_mine[i]) && again[i].u == e_mine[i].u;
                size_t ma = 0, mb = 0;
                for (size_t p = 0; ok && p < L; ++p) { ma = std::max(ma, again[i].l[p]); mb = std::max(mb, e_mine[i].l[p]); ok = ma == mb; }
            }
            if (!ok) { ++bad; std::printf("fold differs (L=%zu, parts=%zu)\n", L, partition.size()); }
        }
    }
    std::printf("%d checks, %d bad\n", checks, bad);
    return bad != 0 || checks < 100;
}
''')
    exe = tmp_path / "f"
    lib = os.path.join(ROOT, "fmindex-collection_b200")
    import fmb200  # noqa: F401
    from fmb200 import build as b
    b.build()
    subprocess.run(["g++", "-std=c++20", "-O1", "-Wno-comment", "-I", os.path.join(ROOT, "include"), str(src), "-L", lib, "-lfmb200",
                    f"-Wl,-rpath,{lib}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 bad" in r.stdout


REF_SRC = "/root/reference/src"


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF_SRC, "fmindex-collection")), reason="needs the reference headers (this container only)")
def test_expand_and_fold_against_the_reference_headers(tmp_path):
    """search_scheme.hpp expand / isValid == the reference's (search_scheme/expand.h:146-180, isValid.h:55-93) for every generator
    and many lengths, and search_pseudo's fold() of an expanded scheme re-expands to exactly the same per-symbol scheme -- i.e. the
    part form handed to the device describes the same search (CPU only: no device call)."""
    src = tmp_path / "e.cpp"
    src.write_text(r'''
#include <fmindex-collection/search_scheme/expand.h>
#include <fmindex-collection/search_scheme/generator/all.h>
#include <fmindex-collection/search_scheme/isValid.h>
#include <cstdio>
#include "fmb200/fmb200.hpp"
namespace rs = fmc::search_scheme;
namespace ms = fmb200::search_scheme;
static ms::Scheme conv(rs::Scheme const& ss) { ms::Scheme r; for (auto const& s : ss) r.push_back(ms::Search{s.pi, s.l, s.u}); return r; }
int main() {
    int checks = 0, bad = 0;
    std::vector<rs::Scheme> schemes;
    for (size_t k = 0; k <= 3; ++k) {
        if (k <= 2) schemes.push_back(rs::generator::optimum(0, k));
        schemes.push_back(rs::generator::h2(k + 2, 0, k));
        schemes.push_back(rs::generator::h2(k + 1, 0, k));
        schemes.push_back(rs::generator::pigeon_opt(0, k));
        schemes.push_back(rs::generator::backtracking(k + 1, 0, k));
        schemes.push_back(rs::generator::suffixFilter(k + 1, 0, k));
    }
    for (auto const& ref : schemes) {
        auto mine = conv(ref);
        ++checks; if (ms::isValid(mine) != rs::isValid(ref)) ++bad;
        for (size_t L : {ref[0].pi.size(), ref[0].pi.size() + 1, size_t{7}, size_t{20}, size_t{50}, size_t{151}}) {
            if (L < ref[0].pi.size()) continue;
            auto e_ref = rs::expand(ref, L);
            auto e_mine = ms::expand(mine, L);
            ++checks; if (conv(e_ref) != e_mine) { ++bad; std::printf("expand differs (L=%zu)\n", L); continue; }
            if (e_mine.empty()) continue;
            // fold back into parts and expand again with the folded partition: must reproduce pi and u exactly, and a lower bound
            // sequence that accepts exactly the same (position, errors) pairs: max over the prefix is what counts (e never decreases)
            auto [folded, partition] = fmb200::search_pseudo::detail_pseudo::fold(e_mine);
            auto again = ms::expand(folded, partition);
            ++checks;
            bool ok = again.size() == e_mine.size() && partition.size() <= 16;
            for (size_t i = 0; ok && i < again.size(); ++i) {
                // the first part may be walked in either direction (expand.h:21-28 derives it from the second part; search_ng26 and
                // the device always walk it to the right): same symbols, same bounds -- compare it as a set
                auto first = [&](ms::Search x) { std::sort(x.pi.begin(), x.pi.begin() + partition[folded[i].pi[0]]); return x.pi; };
                ok = first(again[i]) == first(e_mine[i]) && again[i].u == e_mine[i].u;
                size_t ma = 0, mb = 0;
                for (size_t p = 0; ok && p < L; ++p) { ma = std::max(ma, again[i].l[p]); mb = std::max(mb, e_mine[i].l[p]); ok = ma == mb; }
            }
            if (!ok) { ++bad; std::printf("fold differs (L=%zu, parts=%zu)\n", L, partition.size()); }
        }
    }
    std::printf("%d checks, %d bad\n", checks, bad);
    return bad != 0;
}
''')
    exe = tmp_path / "e"
    lib = os.path.join(ROOT, "fmindex-collection_b200")
    import fmb200  # noqa: F401
    from fmb200 import build as b
    b.build()
    # the reference's headers need C++23 and mmser / libsais stand-ins only for the index types, which are not included here
    subprocess.run(["g++", "-std=c++23", "-O1", "-Wno-comment", "-I", os.path.join(ROOT, "include"), "-I", REF_SRC, "-I", os.path.join(ROOT, "oracle", "shim"),
                    str(src), "-L", lib, "-lfmb200", f"-Wl,-rpath,{lib}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 bad" in r.stdout
