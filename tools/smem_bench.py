"""SMEM search (fmb_search_smems, min_len 19) and locate of its SMEMs (fmb_locate_smems, max_occ 500) on the 3 Gbp synthetic index of
bench.py (same generator, seed 3, sampling rate 16, bidirectional), 10 M x 150-symbol reads in four sets:
  errors4   reads with 0-4 planted edits (fmb_synth_reads_err_device, edit distance)
  errors12  the same with up to 12 edits
  foreign   150-symbol windows of a text drawn with another generator (numpy, seed 7; the library's generator with another seed gives
            the same sequence shifted): short SMEMs (about log_4 n symbols) starting almost everywhere
  exact     reads copied from the text (bench.py's exact workload): one SMEM per read
Each set runs once on an image with the text check tables and once on one built under FMB_NO_TEXTCHECK (the images are built one
after the other: two do not fit).  Per run: resident ms per call (CUDA events, warm-up calls first), SMEMs, extensions and line
requests per read, requests per second over the occurrence-block gather ceiling measured in the same run, and the certificate of
tools/smem_certificate.py on the first 100 k reads (from a min_len 0 call; the timed min_len 19 output must be its filtered subset).
Prints one JSON line with the GPU name and power limit.

    python tools/smem_bench.py [--steps 5] [--warmup 2] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FMB_GATHER_OCC_BLOCK = 1


def timed(stream, torch, steps, warmup, call):
    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        res = call()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--text", type=float, default=3e9)
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--certify", type=int, default=100_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import fmb200 as fmb
    from fmb200 import capi
    from tools.smem_certificate import certify
    if fmb.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    n, nq, L = int(args.text), args.reads, 150
    nc = min(args.certify, nq)
    off = np.arange(nq + 1, dtype=np.uint64) * np.uint64(L)
    out = {"gpu": gpu, "n": n, "reads": nq, "read_len": L, "min_len": 19, "max_occ": 500, "certified_reads": nc, "runs": []}
    stream = torch.cuda.current_stream()
    for text_check in (True, False):
        if text_check:
            os.environ.pop("FMB_NO_TEXTCHECK", None)
        else:
            os.environ["FMB_NO_TEXTCHECK"] = "1"
        d_text = capi.synth_text_device(0, 5, n, 3)
        index = fmb.Index.build_from_device_text(5, d_text, n, sampling_rate=16, bidirectional=True, device=0)
        os.environ.pop("FMB_NO_TEXTCHECK", None)
        capi.index_set_stream(index, stream.cuda_stream)
        sets = {}
        for name, me in (("errors4", 4), ("errors12", 12)):
            d = capi.synth_reads_err_device(0, d_text, n, nq, L, 4, 5, me, True)
            sets[name] = np.zeros(nq * L, dtype=np.uint8)
            capi.copy_to_host(0, sets[name], d, nq * L)
            capi.device_free(0, d)
        d = capi.synth_reads_device(0, d_text, n, nq, L, 4)
        sets["exact"] = np.zeros(nq * L, dtype=np.uint8)
        capi.copy_to_host(0, sets["exact"], d, nq * L)
        capi.device_free(0, d)
        capi.device_free(0, d_text)
        rng = np.random.default_rng(7)
        other = rng.integers(1, 5, size=100_000_000, dtype=np.uint8)
        starts = rng.integers(0, other.size - L, size=nq)
        sets["foreign"] = np.empty(nq * L, dtype=np.uint8)
        for lo in range(0, nq, 1 << 20):
            hi = min(nq, lo + (1 << 20))
            sets["foreign"][lo * L:hi * L] = other[starts[lo:hi, None] + np.arange(L)].reshape(-1)
        del other, starts
        ceiling, _, _ = capi.measure_gather(index, FMB_GATHER_OCC_BLOCK)
        info = index.info
        for name, sym in sets.items():
            q = index.upload(sym, off)
            s_ms, res = timed(stream, torch, args.steps, args.warmup, lambda: index.search_smems(q, min_len=19))
            l_ms, loc = timed(stream, torch, args.steps, args.warmup, lambda: index.locate_smems(res, max_occ=500))
            st, lst = res.stats, loc.stats
            timed_smems = res.smems()
            n_smems, n_rows = len(res), len(loc)
            del loc
            qc = index.upload(sym[: nc * L], off[: nc + 1])
            r0 = index.search_smems(qc, min_len=0)
            all_smems = r0.smems()
            st0 = r0.stats
            ok = bool(certify(index, sym[: nc * L], off[: nc + 1], all_smems))
            want = all_smems[(all_smems["end"] - all_smems["begin"]) >= 19]
            ok = ok and bool(np.array_equal(timed_smems[timed_smems["qidx"] < nc], want))
            reqs = st.occ_lookups + st.line_requests
            out["runs"].append({
                "set": name, "text_check": bool(info.text_tables & 1), "search_ms": s_ms, "search_kernel_ms": st.main_kernel_ms,
                "locate_ms": l_ms, "locate_kernel_ms": lst.main_kernel_ms, "smems_per_read": n_smems / nq, "rows_per_read": n_rows / nq,
                "all_smems_per_read": len(all_smems) / nc, "extensions_per_read": st.extensions / nq, "occ_lookups_per_read": st.occ_lookups / nq,
                "line_requests_per_read": st.line_requests / nq, "extensions_per_read_min_len0": st0.extensions / nc,
                "reads_per_s": nq / (s_ms * 1e-3), "requests_per_s": reqs / (s_ms * 1e-3), "gather_ceiling_per_s": ceiling,
                "of_ceiling": reqs / (s_ms * 1e-3) / ceiling, "certified": ok})
            del res, r0, q, qc
            print(json.dumps(out["runs"][-1]), file=sys.stderr, flush=True)
        index.close()
        del index
    out["certified"] = all(r["certified"] for r in out["runs"])
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
