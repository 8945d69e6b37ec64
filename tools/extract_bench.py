"""Text extraction on the 3 Gbp synthetic index (fmb_synth_text_device, sigma 5, seed 3, sampling rate 16, bidirectional): anchor-table
build time and bytes, whole-text reconstruction and random 150-symbol windows, each rate also as a fraction of the request ceiling
measured in the same run (fmb_measure_gather(FMB_GATHER_JUMP_ENTRY): independent random jump-table entries per second).  Prints one
JSON line.  The text is generated on the device and also kept on the host, so every figure comes with a check of its output.

    python tools/extract_bench.py [--n 3000000000] [--windows 10000000] [--repeat 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_name_and_power():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        return out
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_000_000_000)
    ap.add_argument("--windows", type=int, default=10_000_000)
    ap.add_argument("--length", type=int, default=150)
    ap.add_argument("--repeat", type=int, default=3)
    a = ap.parse_args()

    import fmb200
    from fmb200 import capi
    if fmb200.device_count() < 1:
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    n = a.n
    d_text = capi.synth_text_device(0, 5, n, 3)
    t0 = time.perf_counter()
    index = fmb200.Index.build_from_device_text(5, d_text, n, sampling_rate=16, bidirectional=True, device=0)
    build_s = time.perf_counter() - t0
    text = np.empty(n, dtype=np.uint8)
    capi.copy_to_host(0, text, d_text, n)
    capi.device_free(0, d_text)
    ceiling, _, _ = capi.measure_gather(index, 2)

    # anchor table: built by the first extraction call (one symbol)
    before = index.info.device_bytes
    t0 = time.perf_counter()
    index.extract(0, 0, 1)
    anchor_s = time.perf_counter() - t0
    anchor_bytes = index.info.device_bytes - before
    length = int(index.sequence_lengths()[0])

    # whole text: the counters of one full-sequence range, the time of fmb_index_reconstruct_text (best of --repeat, host clock around
    # a call that ends in a device synchronise; includes the n-byte copy to the host)
    _, st = index.extract(0, 0, length, with_stats=True)
    rec_walk_ms = st.main_kernel_ms
    best = float("inf")
    for _ in range(a.repeat):
        t0 = time.perf_counter()
        out = index.reconstruct_text()
        best = min(best, time.perf_counter() - t0)
    assert np.array_equal(out, text), "reconstructed text differs"
    del out
    rec_requests = st.line_requests + st.lf_steps      # jump-table entries + occurrence blocks read by the walks

    # random windows of --length symbols
    rng = np.random.default_rng(1)
    L = a.length
    b = rng.integers(0, length - L, size=a.windows).astype(np.uint64)
    e = b + np.uint64(L)
    seq = np.zeros(a.windows, dtype=np.uint64)
    import ctypes as C
    out = np.empty(a.windows * L, dtype=np.uint8)
    offsets = np.empty(a.windows + 1, dtype=np.uint64)
    wbest, wst = float("inf"), None
    for _ in range(a.repeat):      # the C call itself: fmb_extract into one preallocated buffer
        s = capi.Stats()
        t0 = time.perf_counter()
        capi._check(capi.lib().fmb_extract(index.h, capi._ptr(seq), capi._ptr(b), capi._ptr(e), C.c_uint64(a.windows), capi._ptr(out),
                                           C.c_uint64(out.size), capi._ptr(offsets), C.byref(s)))
        dt = time.perf_counter() - t0
        if wst is None or s.main_kernel_ms < wst.main_kernel_ms:
            wst = s
        wbest = min(wbest, dt)
    for i in rng.choice(a.windows, 10000, replace=False):
        assert np.array_equal(out[int(offsets[i]):int(offsets[i + 1])], text[int(b[i]):int(e[i])]), "window %d differs" % i
    del out

    res = {
        "gpu": gpu_name_and_power(),
        "n": n, "sampling_rate": 16, "seed": 3,
        "index_build_s": round(build_s, 2),
        "jump_entry_ceiling_requests_per_s": ceiling,
        "anchor_table": {"build_ms": round(anchor_s * 1e3, 1), "bytes": anchor_bytes, "anchors": index.info.n_samples + index.info.n_delims},
        "reconstruct": {
            "call_ms": round(best * 1e3, 1),
            "walk_kernel_ms": round(rec_walk_ms, 2),
            "output_GB_per_s_call": round(n / best / 1e9, 2),
            "output_GB_per_s_walk_kernel": round(n / (rec_walk_ms * 1e-3) / 1e9, 2),
            "jump_requests": st.line_requests, "lf_steps": st.lf_steps,
            "requests_per_16_symbols": round(16 * rec_requests / length, 4),
            "walk_requests_per_s_fraction_of_ceiling": round(rec_requests / (rec_walk_ms * 1e-3) / ceiling, 3),
        },
        "windows": {
            "count": a.windows, "length": L,
            "call_ms": round(wbest * 1e3, 1),
            "walk_kernel_ms": round(wst.main_kernel_ms, 2),
            "windows_per_s_call": round(a.windows / wbest, 0),
            "windows_per_s_walk_kernel": round(a.windows / (wst.main_kernel_ms * 1e-3), 0),
            "requests_per_window": round((wst.line_requests + wst.lf_steps) / a.windows, 3),
            "walk_requests_per_s_fraction_of_ceiling": round((wst.line_requests + wst.lf_steps) / (wst.main_kernel_ms * 1e-3) / ceiling, 3),
        },
    }
    print(json.dumps(res))


if __name__ == "__main__":
    main()
