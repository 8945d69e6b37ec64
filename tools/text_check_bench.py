"""Exact search + locate with and without the text check (FMB_TEXT_CHECK) on ONE 3 Gbp index, alternating the exact modes
FMB_EXACT_AUTO and FMB_EXACT_NO_TEXT round by round, like bench.py's exact workload (10 M x 150 bp reads copied from the text,
sampling rate 16).  Prints one JSON line: per mode and round ms per step, search / locate kernel ms, line requests per read of the
search kernel, plus the GPU name and power limit and the device memory in use after the build and its peak during the build.

    python tools/text_check_bench.py [--rounds 6] [--steps 10] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--text", type=float, default=3e9)
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import fmb200 as fmb
    from fmb200 import capi
    if fmb.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    total = torch.cuda.mem_get_info(0)[1]
    peak = [0]
    done = threading.Event()

    def sample():                     # device memory in use, sampled while the index is built
        while not done.is_set():
            peak[0] = max(peak[0], total - torch.cuda.mem_get_info(0)[0])
            time.sleep(0.02)

    n, nq, L = int(args.text), args.reads, 150
    base = total - torch.cuda.mem_get_info(0)[0]
    th = threading.Thread(target=sample, daemon=True)
    th.start()
    t0 = time.time()
    d_text = capi.synth_text_device(0, 5, n, 3)
    index = fmb.Index.build_from_device_text(5, d_text, n, sampling_rate=16, bidirectional=True, device=0)
    build_s = time.time() - t0
    done.set()
    th.join()
    d_reads = capi.synth_reads_device(0, d_text, n, nq, L, 4)
    sym = capi.PinnedArray(nq * L, np.uint8)
    capi.copy_to_host(0, sym.array, d_reads, nq * L)
    capi.device_free(0, d_reads)
    capi.device_free(0, d_text)
    off = np.arange(nq + 1, dtype=np.uint64) * np.uint64(L)
    stream = torch.cuda.current_stream()
    capi.index_set_stream(index, stream.cuda_stream)
    q = index.upload(sym.array, off)
    info = index.info
    out = {"gpu": gpu, "n": n, "reads": nq, "read_len": L, "build_s": build_s, "image_gb": info.device_bytes / 1e9,
           "text_tables": info.text_tables, "device_used_after_build_gb": (total - torch.cuda.mem_get_info(0)[0]) / 1e9,
           "device_used_before_build_gb": base / 1e9, "device_peak_during_build_gb": peak[0] / 1e9, "rounds": []}
    ref = {}
    for r in range(args.rounds):
        for mode, name in ((0, "text_check"), (3, "lf_jumps")):
            index.set_exact_mode(mode)
            for _ in range(2):
                res = index.search_exact(q)
                loc = index.locate(res)
            del res, loc
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s_ms, l_ms = [], []
            e0.record(stream)
            for _ in range(args.steps):
                res = index.search_exact(q)
                loc = index.locate(res)
                s_ms.append(res.stats.main_kernel_ms)
                l_ms.append(loc.stats.main_kernel_ms)
                st_s, st_l, n_loc = res.stats, loc.stats, len(loc)
            e1.record(stream)
            torch.cuda.synchronize()
            if r == 0:
                ref[name] = (np.sort(res.hits(), order=["qidx"]), np.sort(loc.locs(), order=["qidx", "seq", "pos"]))
            del res, loc
            out["rounds"].append({"round": r, "mode": name, "ms_per_step": e0.elapsed_time(e1) / args.steps,
                                  "search_ms": float(np.mean(s_ms)), "locate_ms": float(np.mean(l_ms)),
                                  "search_requests_per_read": st_s.line_requests / nq, "located_rows": n_loc, "lf_steps": st_l.lf_steps})
    index.set_exact_mode(0)
    a, b = ref["text_check"], ref["lf_jumps"]
    out["identical"] = bool(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]))
    for name in ("text_check", "lf_jumps"):
        ms = [x["ms_per_step"] for x in out["rounds"] if x["mode"] == name]
        out[name] = {"ms_per_step_median": float(np.median(ms)), "ms_per_step_min": min(ms), "ms_per_step_max": max(ms)}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
