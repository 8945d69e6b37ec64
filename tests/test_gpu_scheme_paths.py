"""GPU parity of the k-error search on the paths of run_scheme and its kernels that only switch on at some batch or table size, or
under a knob: the text list sorted by class (> 65 536 items in a text pass), roots in several slabs, warp stacks that spill in text
mode, the second attempt with a larger hit buffer, collections of many short sequences with queries that hold delimiters, and the
paths of an index without some of its optional tables, which the knobs emulate.  Every case compares hits, located rows and
fmb_stats.extensions with the oracle, and asserts from the kernel trace or from the result that it reached the path it is about.

The knobs are read once per process, so those cases run their searches in a child process (FMB_TRACE_SCHEME=1); the child writes
its results to an .npz and the trace to stderr, and the parent compares them with oracle results computed once per module."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from helpers import hits_equal, locs_equal, make_index_pair

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TEXT_SORT_MIN = 65536           # run_scheme sorts the text list by class above this many items

CHILD = r'''
import json, os, sys
sys.path.insert(0, %r)
import numpy as np
import fmb200 as fmb
job = np.load(sys.argv[1])
runs = json.loads(str(job["runs"]))
g = fmb.Index.from_bwt(int(job["sigma"]), job["bwt"], job["bwt_rev"], job["bm"], job["sq"], job["sp"])
q = g.upload(job["sym"], job["off"])
out = {}
for r in runs:
    sch = tuple(np.array(a, dtype=np.uint32) for a in r["scheme"])
    print("[run %%s]" %% r["name"], file=sys.stderr, flush=True)
    res = g.search_scheme(q, sch, r["part"], r["edit"], n=r["n"])
    out[r["name"] + "_hits"] = res.hits()
    out[r["name"] + "_ext"] = np.array([res.stats.extensions], dtype=np.uint64)
    if r["n"] is None and r["locate"]:
        out[r["name"] + "_locs"] = g.locate(res).locs()
np.savez(sys.argv[2], **out)
print("ok")
''' % ROOT

TRACE_RE = re.compile(r"\[fmb scheme\] slab (\d+) pass (\d+) (frontier|text) kernel: [0-9.]+ ms, (.*)$")
FRONTIER_RE = re.compile(r"(\d+) roots \+ (\d+) items in -> (\d+) text, (\d+) back, (\d+) hits so far")
TEXT_RE = re.compile(r"(\d+) items -> (\d+) to the next text list, (\d+) back")


def parse_trace(stderr):
    """{run name: [(kind, slab, pass, fields)]} from the child's stderr: kind "frontier" has (roots, items in, text, back, hits),
    kind "text" has (items, to the next text list, back)"""
    runs, cur = {}, None
    for line in stderr.splitlines():
        if line.startswith("[run "):
            cur = line[5:-1]
            runs[cur] = []
            continue
        m = TRACE_RE.match(line)
        if m and cur is not None:
            kind = m.group(3)
            f = (FRONTIER_RE if kind == "frontier" else TEXT_RE).search(m.group(4))
            assert f, line
            runs[cur].append((kind, int(m.group(1)), int(m.group(2)), tuple(int(x) for x in f.groups())))
    return runs


def run_child(tmp_path, job, env_extra, tag):
    """runs every search of `job` in a fresh process under env_extra; returns (results npz, trace per run)"""
    out = os.path.join(str(tmp_path), "out_%s.npz" % tag)
    env = dict(os.environ, FMB_TRACE_SCHEME="1", **env_extra)
    r = subprocess.run([sys.executable, "-c", CHILD, job, out], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
    return np.load(out), parse_trace(r.stderr)


def write_job(path, o, sigma, sym, off, runs):
    bm, sq, sp = o.samples
    rev = o.bwt_rev
    np.savez(path, sigma=sigma, bwt=o.bwt, bwt_rev=rev, bm=bm, sq=sq, sp=sp, sym=sym, off=off, runs=json.dumps(runs))
    return path


def scheme_run(name, sch, part, edit, n=None, locate=True):
    return {"name": name, "scheme": [np.asarray(a).tolist() for a in sch], "part": [int(x) for x in part], "edit": bool(edit), "n": n,
            "locate": locate}


def same_list(got, exp):
    """hit-limited results, in order (as tests/test_gpu_search_n.py compares them)"""
    got, exp = np.asarray(got), np.asarray(exp)
    return got.shape == exp.shape and all(np.array_equal(got[f].astype(np.uint64), exp[f].astype(np.uint64))
                                          for f in ("qidx", "lb", "lb_rev", "len", "steps", "e"))


class Expected:
    """oracle hits, located rows and extension counts of one workload, per run, computed on first use"""

    def __init__(self, o, sym, off):
        self.o, self.sym, self.off, self.cache = o, sym, off, {}

    def __call__(self, run):
        from oracle.pyoracle import Counters
        key = run["name"]
        if key not in self.cache:
            sch = tuple(np.array(a, dtype=np.uint32) for a in run["scheme"])
            if run["n"] is None:
                ctr = Counters()
                hits = self.o.search_ng26(self.sym, self.off, sch, run["part"], run["edit"], counters=ctr)
                self.cache[key] = (hits, self.o.locate(hits) if run["locate"] else None, int(ctr.extensions))
            else:
                self.cache[key] = (self.o.search_ng26(self.sym, self.off, sch, run["part"], run["edit"], max_hits=run["n"]), None, None)
        return self.cache[key]


def check_runs(res, runs, expected, extensions=True):
    for r in runs:
        hits, locs, ext = expected(r)
        name = r["name"]
        if r["n"] is None:
            assert hits_equal(res[name + "_hits"], hits), name
            if r["locate"]:
                assert locs_equal(res[name + "_locs"], locs), name
            if extensions:
                assert int(res[name + "_ext"][0]) == ext, (name, int(res[name + "_ext"][0]), ext)
        else:
            assert same_list(res[name + "_hits"], hits), name


# ---- b. a large batch on the 1 Mbp index: the text list is sorted by class before the text kernel --------------------------------

NQ_B = 80000
L_B = 100


@pytest.fixture(scope="module")
def wl_b(tmp_path_factory):
    """the 1 Mbp single sequence of test_larger_single_sequence (bidirectional k-mer table k = 8), 80 000 reads of 100 symbols with
    0 / 1 / 2 planted edits, k = 2 optimum scheme, Hamming and edit distance"""
    from fmb200 import schemes, synth
    from oracle.pyoracle import Oracle
    text = synth.text(1 << 20, 5, 1)
    o = Oracle.build(text, 5, 16, True)
    reads, _ = synth.reads_from_text(text, NQ_B, L_B, 41)
    a = NQ_B // 3
    reads[a:2 * a] = synth.plant_errors(reads[a:2 * a], 5, 1, True, 42)
    reads[2 * a:] = synth.plant_errors(reads[2 * a:], 5, 2, True, 43)
    sym, off = synth.flatten(reads)
    sch = schemes.optimum(0, 2)
    part = schemes.uniform_partition(sch[0].shape[1], L_B)
    runs = [scheme_run("edit", sch, part, True), scheme_run("ham", sch, part, False)]
    d = tmp_path_factory.mktemp("wl_b")
    job = write_job(os.path.join(str(d), "job.npz"), o, 5, sym, off, runs)
    return {"o": o, "reads": reads, "sch": sch, "part": part, "runs": runs, "job": job, "exp": Expected(o, sym, off), "dir": d}


def largest_text_pass(trace):
    return max([f[0] for kind, _, _, f in trace if kind == "text"], default=0)


# knob -> the run whose trace must show a text pass above TEXT_SORT_MIN (None: the knob turns text mode off)
KNOBS = [
    ({}, "edit"),
    ({"FMB_NO_TEXT": "1"}, None),
    ({"FMB_NO_SCHEME_JUMP": "1"}, None),            # (no jump tables in the view: no text windows either)
    ({"FMB_NO_BIKMER": "1"}, "edit"),
    ({"FMB_NO_JUMP4": "1"}, "edit"),
]


@pytest.mark.parametrize("env,big_run", KNOBS, ids=[(",".join(e) or "default") for e, _ in KNOBS])
def test_large_batch_and_knobs(wl_b, tmp_path, env, big_run):
    """hits, located rows and extension counts equal the oracle's with the default paths and with every knob that emulates an index
    without some of its optional tables (each is documented to give the same results)"""
    res, trace = run_child(tmp_path, wl_b["job"], env, "b")
    if big_run is None:
        assert all(kind == "frontier" for r in trace.values() for kind, _, _, _ in r), "the knob did not turn text mode off"
    else:
        assert largest_text_pass(trace[big_run]) > TEXT_SORT_MIN, trace[big_run]
    print({r: largest_text_pass(t) for r, t in trace.items()}, {r["name"]: int(res[r["name"] + "_ext"][0]) for r in wl_b["runs"]})
    check_runs(res, wl_b["runs"], wl_b["exp"])


# ---- c. roots in several slabs ---------------------------------------------------------------------------------------------------

NQ_C = 3000


@pytest.fixture(scope="module")
def wl_c(wl_b):
    """the first 3000 reads of workload b: 9000 roots, in slabs of 1009 (a prime: a slab boundary splits the searches of a query)"""
    from fmb200 import synth
    sym, off = synth.flatten(wl_b["reads"][:NQ_C])
    sch, part = wl_b["sch"], wl_b["part"]
    runs = [scheme_run("edit", sch, part, True), scheme_run("ham", sch, part, False)]
    limited = [scheme_run("%s_n%d" % ("edit" if e else "ham", n), sch, part, e, n) for e in (False, True) for n in (1, 3, 10 ** 9)]
    job = write_job(os.path.join(str(wl_b["dir"]), "job_c.npz"), wl_b["o"], 5, sym, off, runs)
    job_n = write_job(os.path.join(str(wl_b["dir"]), "job_c_n.npz"), wl_b["o"], 5, sym, off, runs + limited)
    return {"runs": runs, "limited": limited, "job": job, "job_n": job_n, "exp": Expected(wl_b["o"], sym, off)}


@pytest.mark.parametrize("text", [True, False], ids=["text", "no_text"])
def test_slabs(wl_c, tmp_path, text):
    """FMB_SCHEME_SLAB=1009: text mode (Hamming, edit) or FMB_NO_TEXT, and hit-limited searches (n = 1, 3, 10^9; in order)"""
    env = {"FMB_SCHEME_SLAB": "1009"}
    if not text:
        env["FMB_NO_TEXT"] = "1"
    runs = wl_c["runs"] + (wl_c["limited"] if text else [])
    res, trace = run_child(tmp_path, wl_c["job_n"] if text else wl_c["job"], env, "c")
    for r in runs:
        slabs = {s for _, s, _, _ in trace[r["name"]]}
        print(r["name"], "slabs", len(slabs))
        assert len(slabs) > 1, (r["name"], slabs)
        assert text == any(kind == "text" for kind, _, _, _ in trace[r["name"]]) or r["n"] is not None, r["name"]
    check_runs(res, runs, wl_c["exp"])


# ---- d. warp stacks that spill in text mode ---------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def wl_rep(tmp_path_factory, gpu):
    """the repetitive fixture of test_scheme_search_repetitive_text: 40 copies of a 50-symbol unit with 2 substitutions each,
    60 reads of 30 symbols with one planted error; wide intervals for a long time, so many children per node"""
    from fmb200 import schemes, synth
    from oracle.pyoracle import Oracle
    rng = np.random.default_rng(3)
    unit = rng.integers(1, 5, size=50).astype(np.uint8)
    seqs = []
    for _ in range(40):
        u = unit.copy()
        for p in rng.integers(0, 50, size=2):
            u[p] = rng.integers(1, 5)
        seqs.append(u)
    text = np.concatenate([np.concatenate([s, [0]]) for s in seqs]).astype(np.uint8)
    o = Oracle.build(text, 5, 4, True)
    reads = np.array([seqs[i % 40][5:35] for i in range(60)], dtype=np.uint8)
    sym, off = synth.flatten(synth.plant_errors(reads, 5, 1, True, 4))          # searched with both distances
    runs = []
    for k in (1, 2):
        sch = schemes.optimum(0, k)
        part = schemes.uniform_partition(sch[0].shape[1], 30)
        runs += [scheme_run("edit_k%d" % k, sch, part, True), scheme_run("ham_k%d" % k, sch, part, False)]
    d = tmp_path_factory.mktemp("wl_rep")
    job = write_job(os.path.join(str(d), "job.npz"), o, 5, sym, off, runs)
    return {"runs": runs, "job": job, "exp": Expected(o, sym, off), "spill": ()}


@pytest.fixture(scope="module")
def wl_d(wl_b):
    """every 10th read of workload b, with its k = 2 optimum scheme (whose roots reach the text list in step: they never spill, even
    at 33 items per stack) and with a one-part k = 1 scheme, which branches from the root on while the intervals are wide"""
    from fmb200 import schemes, synth
    sym, off = synth.flatten(wl_b["reads"][::10])
    sch, part = wl_b["sch"], wl_b["part"]
    bt = schemes.backtracking(1, 0, 1)
    runs = [scheme_run("edit", sch, part, True), scheme_run("ham", sch, part, False),
            scheme_run("bt_edit", bt, [L_B], True), scheme_run("bt_ham", bt, [L_B], False)]
    job = write_job(os.path.join(str(wl_b["dir"]), "job_d.npz"), wl_b["o"], 5, sym, off, runs)
    return {"runs": runs, "job": job, "exp": Expected(wl_b["o"], sym, off), "spill": ("bt_edit", "bt_ham")}


@pytest.mark.parametrize("cap", [33, 64])
@pytest.mark.parametrize("workload", ["b", "rep"])
def test_spilled_stacks_in_text_mode(wl_d, wl_rep, tmp_path, cap, workload):
    """FMB_SCHEME_CAP = 33 / 64 items per warp stack: the frontier kernel spills whole rounds of children to the overflow list while
    it also stages text-class items (the refill must flush them when they alone block it)"""
    wl = wl_d if workload == "b" else wl_rep
    res, trace = run_child(tmp_path, wl["job"], {"FMB_SCHEME_CAP": str(cap)}, "d")
    spilled = {}
    for r in wl["runs"]:
        t = trace[r["name"]]
        assert any(kind == "text" for kind, _, _, _ in t), r["name"]              # text mode
        # the first frontier pass of a slab runs before any text pass: what it sends back can only be spills
        spilled[r["name"]] = sum(f[3] for kind, _, p, f in t if kind == "frontier" and p == 0)
    print(spilled)
    assert all(spilled[name] > 0 for name in wl["spill"]) and sum(spilled.values()) > 0, spilled
    check_runs(res, wl["runs"], wl["exp"])


def test_stack_cap_out_of_range_is_refused(gpu, tmp_path):
    """a warp stack below 32 items (or not a number, which atoi would read as 0) could never take a round of roots, and one whose
    block exceeds the shared memory cannot launch: the search fails with FMB_EINVAL before any launch"""
    code = r'''
import sys
sys.path.insert(0, %r)
import numpy as np
import fmb200 as fmb
from fmb200 import schemes, synth
text = synth.multi_text([3000], 5, 2)
from oracle.pyoracle import Oracle
o = Oracle.build(text, 5, 8, True)
g = fmb.Index.from_bwt(5, o.bwt, o.bwt_rev, *o.samples)
reads, _ = synth.reads_from_text(text[:3001], 50, 20, 1)
q = g.upload(*synth.flatten(reads))
sch = schemes.optimum(0, 1)
for n in (None, 5):
    launches = fmb.capi.kernel_launch_count()
    try:
        g.search_scheme(q, sch, schemes.uniform_partition(2, 20), True, n=n)
        raise SystemExit("accepted")
    except fmb.FmbError as e:
        assert e.code == -1 and "FMB_SCHEME_CAP" in str(e), str(e)
    assert fmb.capi.kernel_launch_count() == launches, "a kernel ran"
print("refused")
''' % ROOT
    for bad in ("0", "31", "100000", "abc"):
        r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, FMB_SCHEME_CAP=bad), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0 and "refused" in r.stdout, (bad, r.stdout[-2000:] + r.stderr[-2000:])


# ---- a. many short sequences, queries that straddle delimiters ------------------------------------------------------------------

@pytest.mark.parametrize("sigma", [5, 21])
def test_short_sequences_and_flagged_queries(gpu, sigma):
    """a few hundred sequences of 1..200 symbols (a quarter shorter than 16), reads from the whole concatenation: some straddle one or
    more delimiters and hold symbol 0 (DNA: flagged queries, no k-mer lookup, no jumps, no text class), in one batch with
    ordinary reads; rows whose window meets a delimiter within 16 symbols go back to the frontier kernel (`notext`)"""
    from fmb200 import schemes, synth
    from oracle.pyoracle import Counters
    rng = np.random.default_rng(7 + sigma)
    lens = np.concatenate([rng.integers(1, 16, size=100), rng.integers(16, 201, size=300)])
    rng.shuffle(lens)
    text = synth.multi_text(lens.tolist(), sigma, 31)
    o, g = make_index_pair(gpu, text, sigma, 4)
    L = 24
    start = rng.integers(0, text.size - L, size=1500)
    reads = text[start[:, None] + np.arange(L)[None, :]]
    reads[750:1125] = synth.plant_errors(reads[750:1125], sigma, 1, True, 8)
    sym, off = synth.flatten(reads)
    flagged = (reads == 0).any(axis=1)
    assert 100 < flagged.sum() < len(reads) - 100                          # both kinds in the batch
    q = g.upload(sym, off)
    near_end = 0
    for k in (1, 2):
        sch = schemes.optimum(0, k)
        part = schemes.uniform_partition(sch[0].shape[1], L)
        for edit in (False, True):
            ctr = Counters()
            exp = o.search_ng26(sym, off, sch, part, edit, counters=ctr)
            res = g.search_scheme(q, sch, part, edit)
            assert hits_equal(res.hits(), exp), (k, edit)
            locs = g.locate(res).locs()
            exp_locs = o.locate(exp)
            assert locs_equal(locs, exp_locs), (k, edit)
            assert res.stats.extensions == ctr.extensions, (k, edit, res.stats.extensions, ctr.extensions)
            assert np.isin(exp["qidx"], np.flatnonzero(flagged)).any() and np.isin(exp["qidx"], np.flatnonzero(~flagged)).any()
            # located rows whose text reaches the sequence end within the read plus 16 symbols
            near_end += int(np.sum(lens[locs["seq"].astype(np.int64)] - locs["pos"].astype(np.int64) < L + 16))
    assert near_end > 0


# ---- e. more hits than the first hit buffer holds --------------------------------------------------------------------------------

def test_hit_buffer_second_attempt(tmp_path):
    """4000 copies of a 120-symbol unit with 3 substitutions each, 3000 reads of 30 symbols from the unit: the unlimited k = 2 search
    reports more hits than max(2^20, 8 nq), the size of the first attempt's buffer, so run_scheme runs again with the counted size;
    with n = 10^9 the ordered path does the same before it sorts.  (Roots in slabs of 509: with hundreds of single-row paths per
    root, the text lists of larger slabs exceed their capacity, which the search reports as FMB_EOVERFLOW.)"""
    from fmb200 import schemes, synth
    from oracle.pyoracle import Oracle
    rng = np.random.default_rng(5)
    U, C, L, nq = 120, 4000, 30, 3000
    unit = rng.integers(1, 5, size=U).astype(np.uint8)
    cop = np.tile(unit, (C, 1))
    for c in range(C):
        p = rng.integers(0, U, size=3)
        cop[c, p] = 1 + (cop[c, p] - 1 + rng.integers(1, 4, size=3)) % 4
    text = np.concatenate([cop.reshape(-1), [0]]).astype(np.uint8)
    o = Oracle.build(text, 5, 16, True)
    st = rng.integers(0, U - L, size=nq)
    sym, off = synth.flatten(unit[st[:, None] + np.arange(L)[None, :]])
    sch = schemes.optimum(0, 2)
    part = schemes.uniform_partition(sch[0].shape[1], L)
    runs = [scheme_run(("edit" if e else "ham") + ("_n" if n else ""), sch, part, e, n, locate=False) for e in (False, True) for n in (None, 10 ** 9)]
    exp = Expected(o, sym, off)
    for r in runs:
        if r["n"] is None:
            print(r["name"], "hits", len(exp(r)[0]), "first buffer", max(1 << 20, 8 * nq))
            assert len(exp(r)[0]) > max(1 << 20, 8 * nq), r["name"]
    res, trace = run_child(tmp_path, write_job(os.path.join(str(tmp_path), "job.npz"), o, 5, sym, off, runs), {"FMB_SCHEME_SLAB": "509"}, "e")
    for r in runs:
        assert sum(1 for kind, slab, p, _ in trace[r["name"]] if kind == "frontier" and slab == 0 and p == 0) == 2, r["name"]   # two attempts
    check_runs(res, runs, exp)
