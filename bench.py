#!/usr/bin/env python
"""bench.py -- benchmark of the FM-index hot path on B200 (BASELINE.json: "queries/s (150bp, k=0/1/2, 3Gbp index)").

  python bench.py --gpus N --steps K --warmup W        our arm (libfmb200.so, hand-written sm_100a CUDA).  Default workload "all":
                                                       ONE 3 Gbp index per GPU, then five workloads on it -- exact search + locate
                                                       (BASELINE configs[1], the headline of the JSON line) and the k = 1 / k = 2
                                                       optimum search schemes with Hamming and edit distance (configs[2]) -- each
                                                       with its own resident value, end-to-end value, roofline and parity check
                                                       (`workloads` object of the line).
  python bench.py --workload k2-edit | locate-heavy | protein-k1-hamming | c1 | repeat150 ...   one workload (the other configs)
  python bench.py --scaling strong --gpus N ...        the 10 M reads are split over the N ranks (default: weak, 10 M per rank)
  python bench.py --impl reference ...                 reference arm: the reference's own CPU search + locate on the host cores
                                                       (oracle/_ref/libfmref.so, all host threads), bounded sample per step

One "step" = one pass of search + locate over the whole read batch of a workload.  `value` = queries/s with the reads already
resident in HBM (CUDA events on the launching stream); `e2e` = the same through the C-ABI call fmb_search_and_locate with HOST
buffers (pinned), H2D and D2H inside the timed region.  Multi GPU (torchrun, one rank per GPU): the index is replicated per GPU,
the reads are sharded, no collective on the data path; the only collectives are barriers and the max-over-ranks of the times.

roofline.frac is PHYSICAL: requests issued by the kernel x 128 B (the DRAM line a random request moves; cross-checked with ncu
dram__bytes, profiles/) / kernel time / measured HBM peak.  The reference algorithm's work (occ-block lookups x 32 B, SURVEY.md
section 8d) is reported next to it as `algorithmic_*`; `algorithmic_speedup` = algorithmic GB/s / peak may exceed 1 because the
kernels answer many lookups with one request.  The random-request ceiling of the device is measured IN THIS RUN over the index's
own tables (fmb_measure_gather).

Sizes can be reduced for smoke runs with --text / --reads / --read-len (the JSON line then names the reduced workload).

--dump-outputs DIR writes what the last timed step returned (the hits of the search and the rows of locate) as .npy files, so that
two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LINE_BYTES = 128.0     # DRAM bytes moved by one random request (profiles/r01_ncu_full_exact2_locate.txt: 116 B per 32-B lookup)
DUMP_QUERIES = 1 << 14                # --dump-outputs: queries in the fixed sample whose results are written
DUMP_BYTES = 64 << 20                 # --dump-outputs: upper bound of all files together


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)"""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DNA_SET = ("exact", "k1-hamming", "k1-edit", "k2-hamming", "k2-edit")
WORKLOADS = ("all",) + DNA_SET + ("locate-heavy", "protein-k1-hamming", "protein-k1-edit", "c1", "repeat150")


def family_of(wl):
    """text family a workload runs on: workloads of one family share one index"""
    if wl.startswith("protein"):
        return "protein"
    if wl in ("locate-heavy", "repeat150"):
        return "repeat"
    return "dna"


def scheme_of(wl, L):
    """(scheme, partition, edit, k) of a workload: optimum(0,k) with a uniform partition (BASELINE configs[2]); exact: None"""
    from fmb200 import schemes
    if "-k" not in "-" + wl:
        return None, None, False, 0
    k = int(wl.split("k")[1][0])
    sch = schemes.optimum(0, k)
    return sch, schemes.uniform_partition(sch[0].shape[1], L), wl.endswith("edit"), k


def describe(wl, nq, L, n_text, sigma, rate, k, edit, per):
    protein = sigma > 5
    unit = "aa" if protein else "bp"
    if wl in ("exact", "c1"):
        what, src = "exact search + locate", "reads copied from the text"
    elif wl == "locate-heavy":
        what, src = "exact search + locate of repeat-family 20-mers (many hits per read)", "windows of a 1 kbp unit present in 1000 copies"
    elif wl == "repeat150":
        what, src = "exact search + locate of repeat-family 150-mers (intervals stay wide: ~200 copies match each read)", "windows of a 1 kbp unit present in 1000 copies"
    else:
        what = f"k<={k} {'edit' if edit else 'hamming'} search (optimum scheme, uniform partition) + locate"
        src = f"reads copied from the text with 0..{k} planted {'edits' if edit else 'substitutions'} each"
    return (f"{what}, {nq} x {L}{unit} {src}, synthetic {n_text} {unit} {'protein' if protein else 'DNA'} BiFMIndex (sigma {sigma}, "
            f"sampling rate {rate}), {per}")


def make_reads(capi, device, wl, d_text, n_text, nq, L, seed, read_seed, sigma):
    """synthetic reads of a workload on the device -> pinned host arrays (symbols, offsets)"""
    sch, _, edit, k = scheme_of(wl, L)
    if wl in ("exact", "c1"):
        d_reads = capi.synth_reads_device(device, d_text, n_text, nq, L, read_seed)
    elif wl in ("locate-heavy", "repeat150"):
        d_reads = capi.synth_unit_reads_device(device, 5, nq, L, seed, 1000)      # windows of the repeat unit (unit = f(seed))
    else:
        d_reads = capi.synth_reads_err_device(device, d_text, n_text, nq, L, read_seed, sigma, k, edit)
    sym = capi.PinnedArray(nq * L, np.uint8)
    capi.copy_to_host(device, sym.array, d_reads, nq * L)
    capi.device_free(device, d_reads)
    off = capi.PinnedArray(nq + 1, np.uint64)
    off.array[:] = np.arange(nq + 1, dtype=np.uint64) * np.uint64(L)
    return sym, off


def reference_index(index, sigma=5):
    """host-side reference index over exactly the same BWT bytes and samples (BiFMIndex(bwt, bwtRev, SparseArray))"""
    from oracle.pyoracle import Ref
    t0 = time.time()
    bwt, rev, bm, sq, sp = index.export()
    t1 = time.time()
    ref = Ref.from_bwt(sigma, bwt, rev, bm, sq, sp)
    log(f"reference index: export {t1 - t0:.1f}s, construct {time.time() - t1:.1f}s")
    return ref


def cpu_search_locate(ref, sym, off, b, e, threads, L, scheme=None, partition=None, edit=False, want_locs=False):
    """the reference's search (search_no_errors::search or search_ng26::search<Edit> with the given scheme) + LocateLinear on
    reads [b,e), queries sharded over `threads` std::threads; returns (seconds, n_located[, located rows])"""
    s = sym[b * L: e * L]
    o = (off[b: e + 1] - off[b]).astype(np.uint64)
    hits = ref.search_exact(s, o, threads=threads) if scheme is None else ref.search_ng26(s, o, scheme, partition, edit, threads=threads)
    t = ref.last_seconds
    locs = ref.locate(hits, threads=threads)
    t += ref.last_seconds
    return (t, len(locs), locs) if want_locs else (t, len(locs))


def ref_name_of(scheme, edit, k):
    return "search_no_errors::search (batched)" if scheme is None else f"search_ng26::search<{'true' if edit else 'false'}>(optimum(0,{k}))"


def output_sample(res, loc, nq, max_bytes):
    """what one step returned, for --dump-outputs: the hits and located rows of a fixed, seeded sample of the queries as float64
    arrays (one column per field, exact below 2^53), sorted by all fields because the device reports them in an order that depends
    on scheduling; each array is cut to `max_bytes`.  `counts` = rows of the whole output (hits, located rows)."""
    sample = np.random.default_rng(0).choice(nq, size=min(nq, DUMP_QUERIES), replace=False).astype(np.uint64)
    out = {"counts": np.array([len(res), len(loc)], dtype=np.float64)}
    for name, rec in (("hits", res.hits()), ("locs", loc.locs())):
        rec = np.sort(rec[np.isin(rec["qidx"], sample)], order=list(rec.dtype.names))
        arr = np.stack([rec[f].astype(np.float64) for f in rec.dtype.names], axis=1)
        out[name] = arr[: max_bytes // (arr.itemsize * arr.shape[1])]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=WORKLOADS,
                    help="all = exact (BASELINE configs[1], the headline) + k1/k2 hamming/edit (configs[2]) on one index; c1 = configs[0]; "
                         "locate-heavy = configs[3]; protein-* = configs[4]; repeat150 = 150-mers on the repeat-family text")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: --reads is the TOTAL over all ranks")
    ap.add_argument("--text", type=float, default=None, help="text length in symbols (default 3 Gbp; 1 Gaa for protein; 4 Mbp for c1)")
    ap.add_argument("--reads", type=float, default=None, help="reads per GPU (default 10 M; 250 k for locate-heavy; 1 M protein; 100 k c1)")
    ap.add_argument("--read-len", type=int, default=None, help="default 150 (20 for locate-heavy, 50 protein, 100 c1)")
    ap.add_argument("--rate", type=int, default=16)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the headline cpu_baseline sample (the other workloads get a third)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--image-gb", type=float, default=0.0, help="HBM budget of the index image in GB (fmb_set_image_budget; 0 = every table that fits)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the hits and located rows of the last timed step (fixed sample of the queries, float64) to DIR/<workload>_*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: use it with --impl ours")

    wls = list(DNA_SET) if args.workload == "all" else [args.workload]
    head = wls[0]
    fam = family_of(head)
    protein = fam == "protein"
    sigma = 21 if protein else 5
    n_text = int(args.text) if args.text else (1_000_000_000 if protein else (4_000_000 if head == "c1" else 3_000_000_000))
    nq_total = int(args.reads) if args.reads else (250_000 if fam == "repeat" else (1_000_000 if protein else (100_000 if head == "c1" else 10_000_000)))
    L = args.read_len if args.read_len else (20 if head == "locate-heavy" else (50 if protein else (100 if head == "c1" else 150)))
    W = max(args.warmup, 3)
    K = args.steps

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference" and rank != 0:
        return 0
    strong = args.scaling == "strong"
    nq = (nq_total + world - 1) // world if strong else nq_total          # reads of THIS rank
    per = f"{nq_total} reads split over the ranks" if strong else "per GPU"

    # stdout carries exactly ONE line, the JSON result: everything libraries print (NCCL's version banner goes to stdout) is
    # sent to stderr by pointing fd 1 at fd 2 for the duration of the run; the result is written to the saved descriptor
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(result_fd, (json.dumps(line) + "\n").encode())

    # host threads of the pipelined one-call path: the library default (6) assumes the host to itself; with one rank per GPU the
    # ranks share the host cores
    os.environ.setdefault("FMB_E2E_THREADS", str(max(2, min(6, (os.cpu_count() or 6) // max(world, 1)))))

    import torch
    import fmb200 as fmb
    from fmb200 import capi

    if fmb.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: libfmb200 has no CPU fallback")
    device = local_rank
    torch.cuda.set_device(device)
    dist = None
    if world > 1 and args.impl == "ours":
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))

    threads = os.cpu_count() or 1
    metric_head = {"exact": "queries/s (150bp exact search + locate, 3 Gbp index)"}.get(
        head, f"queries/s ({head}, search + locate, {'1 Gaa' if protein else ('4 Mbp' if head == 'c1' else '3 Gbp')} index)")

    if args.image_gb > 0:
        capi.set_image_budget(args.image_gb * 1e9)
    # ---- the SAME text on every rank (the index is replicated per GPU), different reads per rank (queries are sharded) ----------
    t0 = time.time()
    if fam == "repeat":
        d_text = capi.synth_repeat_text_device(device, 5, n_text, 3, 1000, 1000, 10)
    else:
        d_text = capi.synth_text_device(device, sigma, n_text, 3)
    index = fmb.Index.build_from_device_text(sigma, d_text, n_text, sampling_rate=args.rate, bidirectional=True, device=device)
    t1 = time.time()
    data = {}
    for i, wl in enumerate(wls):
        data[wl] = make_reads(capi, device, wl, d_text, n_text, nq, L, 3, 4 + 1000 * rank + 17 * i, sigma)
    capi.device_free(device, d_text)
    log(f"index build {t1 - t0:.1f}s (n={n_text}), reads of {len(wls)} workload(s) {time.time() - t1:.1f}s, device image {index.info.device_bytes / 1e9:.2f} GB")
    tables = index.info.tables
    table_names = [name for bit, name in ((1, "pair"), (2, "kmer"), (4, "jump"), (8, "jump_rev"), (16, "locblock"), (32, "locrow"), (64, "bikmer"),
                                          (128, "jump4"), (256, "jump32")) if tables & bit]

    # ------------------------------------------------------------------------------------------------------
    if args.impl == "reference":
        # the reference's own CPU implementation keeps no device state: the GPU builder only produced the BWT (there is no libsais
        # here); the device image is released BEFORE anything is timed
        ref = reference_index(index, sigma)
        index.close()
        budget = 150.0                              # seconds of CPU work for all W + K steps of all workloads
        share = {wl: (0.5 if wl == head else 0.5 / max(len(wls) - 1, 1)) if len(wls) > 1 else 1.0 for wl in wls}
        out = {}
        for wl in wls:
            sym, off = data[wl]
            scheme, partition, edit, k = scheme_of(wl, L)
            probe = min(nq, 5000 if scheme is not None or fam == "repeat" else 20000)
            t, _ = cpu_search_locate(ref, sym.array, off.array, 0, probe, threads, L, scheme, partition, edit)
            rate_qs = probe / max(t, 1e-9)
            per_step = int(min(nq, max(probe, rate_qs * budget * share[wl] / (W + K))))
            for _ in range(W):
                cpu_search_locate(ref, sym.array, off.array, 0, per_step, threads, L, scheme, partition, edit)
            tot = 0.0
            for _ in range(K):
                t, nloc = cpu_search_locate(ref, sym.array, off.array, 0, per_step, threads, L, scheme, partition, edit)
                tot += t
            qps = per_step * K / tot
            out[wl] = {"value": qps, "unit": "queries/s", "ms_per_step": 1e3 * tot / K,
                       "sample": f"first {per_step} of the {nq} reads per step, {ref_name_of(scheme, edit, k)} + LocateLinear, {threads} threads"}
            log(f"reference {wl}: {qps:.0f} q/s")
        h = out[head]
        line = {"impl": "reference", "metric": metric_head, "value": h["value"], "unit": "queries/s",
                "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": h["ms_per_step"], "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": describe(head, nq, L, n_text, sigma, args.rate, 0, False, per)},
                "cpu_baseline": {"value": h["value"], "unit": "queries/s", "cores": threads, "kind": "reference", "sample": h["sample"]},
                "e2e": {"value": h["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "the repo's GPU builder only synthesised the text and built the BWT handed to the reference's BiFMIndex(bwt, bwtRev, "
                        "SparseArray) constructor; the device image was freed before the timed region, which is std::chrono around the "
                        "reference's unmodified search + LocateLinear inside oracle/_ref/libfmref.so",
                "workloads": out}
        emit(line)
        return 0

    # ------------------------------------------------------------------------------------------------------
    stream = torch.cuda.current_stream()
    capi.index_set_stream(index, stream.cuda_stream)
    peak, peak_src = load_peaks()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- empirical ceilings of this device, measured in this run over the index's own tables (SURVEY.md section 8d) ----------------
    ceilings = {}
    for name, tab in (("pair_line_128B", 0), ("occ_block_32B", 1), ("jump_entry", 2)):
        try:
            rps, tb, rb = capi.measure_gather(index, tab, 1 << 27)
            ceilings[name] = {"requests_per_s": rps, "table_bytes": tb, "request_bytes": rb, "useful_gbs": rps * rb / 1e9}
        except Exception as ex:
            ceilings[name] = {"requests_per_s": None, "note": str(ex)}
    req_ceiling = max([c["requests_per_s"] for c in ceilings.values() if c.get("requests_per_s")] or [0.0]) or None
    # bare pinned H2D copy of one read batch, all ranks at the same time: the ceiling of the end-to-end number
    sym0 = data[head][0]
    h2d_probe = torch.empty(sym0.array.nbytes, dtype=torch.uint8, device="cuda")
    src = torch.from_numpy(sym0.array)
    h2d_probe.copy_(src)
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        h2d_probe.copy_(src)
    torch.cuda.synchronize()
    h2d_s = max_over_ranks((time.perf_counter() - t0) / 3)
    h2d_gbs = sym0.array.nbytes / h2d_s / 1e9
    del h2d_probe, src
    torch.cuda.empty_cache()

    def ncu_traffic(kernel, key):
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                ent = json.load(f)[kernel]
            return ent["traffic_bytes"] if ent["workload"] == key else None
        except Exception:
            return None

    sampler = ClockSampler(device)
    sampler.start()
    launches0 = capi.kernel_launch_count()
    results, e2e_locs = {}, {}
    dumps = {} if args.dump_outputs and rank == 0 else None          # rank 0's reads only
    for wl in wls:
        sym, off = data[wl]
        scheme, partition, edit, k = scheme_of(wl, L)
        queries = index.upload(sym.array, off.array)          # resident in HBM before the timed region

        def search():
            return index.search_exact(queries) if scheme is None else index.search_scheme(queries, scheme, partition, edit)

        def step():
            res = search()
            loc = index.locate(res)
            return res, loc

        alg_lookups, one_symbol_ms = None, None
        if scheme is None:
            # algorithmic work of the reference algorithm on this batch (SURVEY.md section 8d: occ-block lookups of one-symbol
            # steps), counted once, untimed, by the one-symbol kernel; the timed steps use the default kernel
            index.set_exact_mode(1)
            res = index.search_exact(queries)
            alg_lookups = res.stats.occ_lookups
            one_symbol_ms = res.stats.main_kernel_ms
            del res
            index.set_exact_mode(0)

        for _ in range(W):
            res, loc = step()
        n_hits, n_locs = len(res), len(loc)
        del res, loc
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        search_ms, locate_ms, st_s, st_l = [], [], None, None
        for i in range(K):
            res, loc = step()
            search_ms.append(res.stats.main_kernel_ms)
            locate_ms.append(loc.stats.main_kernel_ms)
            st_s, st_l = res.stats, loc.stats
            if i + 1 < K or dumps is None:
                del res, loc
        ev1.record(stream)
        barrier()
        if dumps is not None:
            dumps[wl] = output_sample(res, loc, nq, DUMP_BYTES // (3 * len(wls)))
            del res, loc
        ms_per_step = max_over_ranks(ev0.elapsed_time(ev1)) / K
        q_all = nq_total if strong else nq * world
        value = q_all / (ms_per_step * 1e-3)

        walk = None
        if wl == "locate-heavy":
            # BASELINE configs[3] measures the LF walk: the same step with the walking kernel (FMB_LOCATE_WALK) instead of the
            # precomputed locate shortcut
            index.set_locate_mode(1)
            for _ in range(2):
                res, loc = step()
                del res, loc
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            w_ms = []
            for _ in range(K):
                res, loc = step()
                w_ms.append(loc.stats.main_kernel_ms)
                w_st = loc.stats
                del res, loc
            e1.record(stream)
            barrier()
            walk_step = max_over_ranks(e0.elapsed_time(e1)) / K
            index.set_locate_mode(0)
            wk = float(np.mean(w_ms))
            walk_lines = n_locs * 2 + w_st.lf_steps
            walk = {"kernel": "locate_pair_kernel" if tables & 16 else "locate_kernel", "ms_per_step": walk_step, "value": q_all / (walk_step * 1e-3),
                    "kernel_ms": wk, "located_rows_per_s": n_locs / (wk * 1e-3), "lf_steps_per_row": w_st.lf_steps / max(n_locs, 1),
                    "requests_per_row": walk_lines / max(n_locs, 1), "requests_per_s": walk_lines / (wk * 1e-3),
                    "achieved": walk_lines * LINE_BYTES / (wk * 1e-3) / 1e9, "frac": walk_lines * LINE_BYTES / (wk * 1e-3) / 1e9 / peak}

        # ---- end to end through the C-ABI with host buffers --------------------------------------------------------
        del queries
        out = capi.PinnedArray(max(n_locs, nq) + 1024, capi.LOC32_DTYPE)
        for _ in range(2):
            index.search_and_locate(sym.array, off.array, scheme=scheme, partition=partition, edit=edit, out=out.array)
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            locs, _st = index.search_and_locate(sym.array, off.array, scheme=scheme, partition=partition, edit=edit, out=out.array)
        torch.cuda.synchronize()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        e2e_qps = q_all * K / e2e_s
        h2d = int(_st.h2d_bytes)          # counted by the library from the copies it issued (equal-length batches: the symbols only,
        d2h = int(_st.d2h_bytes)          # the offsets are generated on the device) / the located rows it copied back
        e2e_locs[wl] = (locs.copy(), out)       # `out` is reused below
        # the same call on 2-bit packed host reads (what fmb200/io.hpp produces while parsing FASTA): a quarter of the bytes cross PCIe
        e2e_packed = None
        if sigma <= 5:
            pw = capi.PinnedArray((nq * L + 15) // 16 + 1, np.uint32)
            packed = capi.pack_queries(sym.array, sigma, words=pw.array)          # untimed: done once, by the reader
            for _ in range(2):
                index.search_and_locate(None, off.array, scheme=scheme, partition=partition, edit=edit, out=out.array, packed=packed)
            barrier()
            t0 = time.perf_counter()
            for _ in range(K):
                plocs, _st = index.search_and_locate(None, off.array, scheme=scheme, partition=partition, edit=edit, out=out.array, packed=packed)
            torch.cuda.synchronize()
            pk_s = max_over_ranks(time.perf_counter() - t0)
            e2e_packed = {"value": q_all * K / pk_s, "unit": "queries/s", "h2d_bytes_per_step": int(_st.h2d_bytes),
                          "d2h_bytes_per_step": int(_st.d2h_bytes), "rows_equal_byte_path": int(len(plocs)) == int(len(locs)),
                          "input": "reads 2-bit packed on the host beforehand (fmb_pack_symbols), fmb_search_and_locate_packed"}
            pw.free()

        # ---- roofline of the dominant kernel (physical; see the module docstring) -------------------------------------------------
        k_ms = float(np.mean(search_ms))
        l_ms = float(np.mean(locate_ms))
        shortcut = bool(tables & 32)
        loc_alg = n_locs * 2 + st_l.lf_steps * 2       # per row: marker test + sample fetch, per LF step: occ block + marker word
        loc_req = 2 * n_locs if shortcut else (2 * n_locs + st_l.lf_steps)
        locate_info = {"kernel": "locate_shortcut_kernel" if shortcut else ("locate_pair_kernel" if tables & 16 else "locate_kernel"),
                       "kernel_ms": l_ms, "lf_steps_per_row": st_l.lf_steps / max(n_locs, 1),
                       "requests_per_row": loc_req / max(n_locs, 1), "requests_per_s": loc_req / (l_ms * 1e-3) if l_ms else None,
                       "achieved": loc_req * LINE_BYTES / (l_ms * 1e-3) / 1e9 if l_ms else None,
                       "frac": loc_req * LINE_BYTES / (l_ms * 1e-3) / 1e9 / peak if l_ms else None,
                       "algorithmic_bytes_per_launch": loc_alg * 32.0,
                       "algorithmic_speedup": loc_alg * 32.0 / (l_ms * 1e-3) / 1e9 / peak if l_ms else None}
        if scheme is None:
            kernel = "exact_search2_kernel" if tables & 1 else "exact_search_kernel"
            alg_bytes = alg_lookups * (64.0 if protein else 32.0)
            ext_per_q = None
        else:
            kernel = "scheme_search_kernel + scheme_text_kernel"      # frontier kernel + text kernel, all launches of one search call
            alg_bytes = st_s.occ_lookups * (64.0 if protein else 32.0)       # SURVEY.md section 8d: 64 B per lookup for sigma = 21
            alg_lookups = st_s.occ_lookups
            ext_per_q = st_s.extensions / nq
        requests = st_s.line_requests
        phys_bytes = requests * LINE_BYTES
        achieved = phys_bytes / (k_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": ncu_traffic(kernel + ":" + wl, f"{nq} x {L} on {n_text}"), "peak_source": peak_src,
                    "kernel_ms": k_ms, "bytes_per_launch": phys_bytes, "requests_per_query": requests / nq,
                    "requests_per_s": requests / (k_ms * 1e-3), "request_ceiling_per_s": req_ceiling,
                    "frac_of_request_ceiling": (requests / (k_ms * 1e-3) / req_ceiling) if req_ceiling else None,
                    "algorithmic_bytes_per_launch": alg_bytes, "algorithmic_lookups_per_query": alg_lookups / nq,
                    "algorithmic_speedup": alg_bytes / (k_ms * 1e-3) / 1e9 / peak,
                    "note": "frac = requests x 128 B / kernel time / peak (physical); algorithmic_speedup = the reference algorithm's occ-block "
                            "lookups x 32 B / kernel time / peak (can exceed 1: one request answers many lookups)",
                    "locate_kernel": locate_info}
        if ext_per_q is not None:
            roofline["extensions_per_query"] = ext_per_q
            roofline["frontier_peak_items_per_warp"] = st_s.frontier_peak
        if one_symbol_ms is not None:
            roofline["one_symbol_kernel_ms"] = one_symbol_ms
        if wl == "locate-heavy":
            # configs[3] is about locate: lead with the WALKING kernel, keep the search kernel's figures as search_kernel
            roofline = {"bound": "hbm", "kernel": walk["kernel"], "achieved": walk["achieved"], "peak": peak, "unit": "GB/s", "frac": walk["frac"],
                        "traffic": None, "peak_source": peak_src, "kernel_ms": walk["kernel_ms"], "located_rows_per_s": walk["located_rows_per_s"],
                        "lf_steps_per_row": walk["lf_steps_per_row"], "requests_per_row": walk["requests_per_row"],
                        "requests_per_s": walk["requests_per_s"], "request_ceiling_per_s": req_ceiling,
                        "shortcut": {**locate_info, "ms_per_step": ms_per_step, "value": value, "located_rows_per_s": n_locs / (l_ms * 1e-3)},
                        "search_kernel": {k2: roofline[k2] for k2 in ("kernel", "kernel_ms", "requests_per_query", "frac")}}
        results[wl] = {"metric": f"queries/s ({wl}, search + locate)", "value": walk["value"] if walk else value, "unit": "queries/s",
                       "ms_per_step": walk["ms_per_step"] if walk else ms_per_step,
                       "kernel_ms": {"search": k_ms, "locate": walk["kernel_ms"] if walk else l_ms},
                       "workload": describe(wl, nq, L, n_text, sigma, args.rate, k, edit, per),
                       "hits_per_step": n_hits, "located_rows_per_step": n_locs, "roofline": roofline,
                       "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                               "frac_of_h2d_ceiling": (e2e_qps / world if not strong else e2e_qps * nq / nq_total) / (nq / (h2d / (h2d_gbs * 1e9)))}}
        if e2e_packed:
            results[wl]["e2e_packed"] = e2e_packed
        log(f"{wl}: resident {results[wl]['value'] / 1e6:.1f} M q/s ({ms_per_step:.2f} ms/step, search kernel {k_ms:.2f} ms, locate {l_ms:.2f} ms), "
            f"e2e {e2e_qps / 1e6:.1f} M q/s" + (f" (packed {e2e_packed['value'] / 1e6:.1f})" if e2e_packed else "") + f", frac {roofline['frac']:.3f}")
    # ---- strong scaling (N > 1, default weak run): ONE batch of nq reads split over the ranks -- rank r searches the reads
    #      [r * nq / N, (r + 1) * nq / N) of its batch; value = nq / max-over-ranks time (BASELINE configs[2]: "sharded queries")
    strong_rows = None
    if world > 1 and not strong:
        strong_rows = {}
        lo, hi = rank * nq // world, (rank + 1) * nq // world
        for wl in wls:
            sym, off = data[wl]
            scheme, partition, edit, k = scheme_of(wl, L)
            ssym = sym.array[lo * L: hi * L]
            soff = (off.array[lo: hi + 1] - off.array[lo]).astype(np.uint64)
            queries = index.upload(ssym, soff)

            def sstep():
                res = index.search_exact(queries) if scheme is None else index.search_scheme(queries, scheme, partition, edit)
                loc = index.locate(res)
                return len(loc)
            sstep()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(K):
                sstep()
            e1.record(stream)
            barrier()
            s_ms = max_over_ranks(e0.elapsed_time(e1)) / K
            del queries
            out = e2e_locs[wl][1]
            index.search_and_locate(ssym, soff, scheme=scheme, partition=partition, edit=edit, out=out.array)
            barrier()
            t0 = time.perf_counter()
            for _ in range(K):
                index.search_and_locate(ssym, soff, scheme=scheme, partition=partition, edit=edit, out=out.array)
            torch.cuda.synchronize()
            s_e2e = max_over_ranks(time.perf_counter() - t0) / K
            strong_rows[wl] = {"reads_total": nq, "reads_per_rank": hi - lo, "ms_per_step": s_ms, "value": nq / (s_ms * 1e-3),
                               "e2e": nq / s_e2e, "unit": "queries/s"}
            log(f"{wl} strong scaling ({nq} reads over {world} ranks): resident {nq / (s_ms * 1e-3) / 1e6:.1f} M q/s, e2e {nq / s_e2e / 1e6:.1f} M q/s")
    launches = capi.kernel_launch_count() - launches0
    clocks = sampler.stop()
    clocks["window"] = "warm-up + timed steps + e2e loops of all workloads"
    if dumps is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for wl, arrays in dumps.items():
            for name, arr in arrays.items():
                np.save(os.path.join(args.dump_outputs, f"{wl}_{name}.npy"), arr)

    h = results[head]
    line = {"metric": metric_head, "value": h["value"], "unit": "queries/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": h["ms_per_step"], "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": h["workload"],
                       "l2_policy": "inputs larger than L2 (index image %.1f GB, reads %.2f GB per workload)" % (index.info.device_bytes / 1e9, nq * L / 1e9),
                       "index_tables": table_names, "image_budget_gb": args.image_gb or None, "image_gb": index.info.device_bytes / 1e9, "hits_per_step": h["hits_per_step"], "located_rows_per_step": h["located_rows_per_step"],
                       "workloads_in_this_line": wls},
            "roofline": h["roofline"], "e2e": h["e2e"], "gpu_launches": launches, "clocks": clocks,
            "ceilings": {"random_requests": ceilings, "request_ceiling_per_s": req_ceiling,
                         "pinned_h2d_gbs_per_gpu_all_ranks_concurrent": h2d_gbs, "ranks": world},
            "workloads": results}
    if strong_rows is not None:
        line["strong_scaling"] = strong_rows

    # ---- CPU baseline + parity: the reference's own search on this box's host cores (rank 0) -------------------------------------
    # N = 1: cpu_baseline (bounded sample, all host threads) + parity on that sample for every workload; N > 1: parity only, on a
    # smaller sample (the other ranks have finished by then)
    if rank == 0 and not args.no_cpu_baseline:
        try:
            ref = reference_index(index, sigma)
            for wl in wls:
                sym, off = data[wl]
                scheme, partition, edit, k = scheme_of(wl, L)
                secs = (args.cpu_seconds if wl == head else args.cpu_seconds / 3.0) * (1.0 if world == 1 else 0.4)
                probe = min(nq, 5000 if scheme is not None or fam == "repeat" else 20000)
                t, _ = cpu_search_locate(ref, sym.array, off.array, 0, probe, threads, L, scheme, partition, edit)
                sample_n = int(min(nq, max(probe, probe / max(t, 1e-9) * secs)))
                t, nloc, exp = cpu_search_locate(ref, sym.array, off.array, 0, sample_n, threads, L, scheme, partition, edit, want_locs=True)
                base = {"value": sample_n / t, "unit": "queries/s", "cores": threads, "kind": "reference",
                        "sample": f"first {sample_n} of the {nq} reads, {ref_name_of(scheme, edit, k)} + LocateLinear, {threads} threads ({t:.1f}s)"}
                if wl == head and world == 1:
                    t1, _ = cpu_search_locate(ref, sym.array, off.array, 0, min(sample_n, probe * 2), 1, L, scheme, partition, edit)
                    base["sample"] += f"; 1 thread: {min(sample_n, probe * 2) / t1:.0f} queries/s"
                # parity on the sample: located rows identical as sorted multisets
                locs = e2e_locs[wl][0]
                got = np.sort(locs[locs["qidx"] < sample_n], order=["qidx", "seq", "pos", "e"])
                exp32 = np.zeros(len(exp), dtype=capi.LOC32_DTYPE)
                for f in ("qidx", "seq", "pos", "e"):
                    exp32[f] = exp[f]
                exp32 = np.sort(exp32, order=["qidx", "seq", "pos", "e"])
                par = {"checked_queries": sample_n, "located_rows": int(len(exp32)), "identical": bool(np.array_equal(got, exp32))}
                results[wl]["parity"] = par
                if world == 1:
                    results[wl]["cpu_baseline"] = base
                log(f"{wl}: cpu {base['value']:.0f} q/s, parity {par}")
            line["parity"] = results[head]["parity"]
            if world == 1:
                line["cpu_baseline"] = results[head]["cpu_baseline"]
        except Exception as ex:   # the baseline must not hide the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "queries/s", "cores": threads, "kind": "reference", "sample": f"failed: {ex}"}
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
