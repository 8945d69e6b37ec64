"""bench.py --workload all with the suffix array (default) and with the locate shortcut it replaces (FMB_NO_SA=1), alternating the
two arms run by run (A B A B A B) so that both see the same state of the machine.  Every run dumps its outputs (--dump-outputs); the
dumps of all runs are compared array for array with the first run's.  Writes one JSON file: the GPU name and power limit, per arm and
run the resident value, ms per step and kernel ms (search, locate) of every workload and the parity objects, and per workload the
medians, the spread between repeats of the same arm and the ratio of the medians.

    python tools/sa_bench.py [--repeats 3] [--steps 20] [--warmup 5] [--out profiles/r05_sa_bench_3gbp_N1.json] [bench.py options]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARMS = (("sa", {}), ("no_sa", {"FMB_NO_SA": "1"}))


def run_bench(extra_env, steps, warmup, dump_dir, passthrough):
    env = dict(os.environ, **extra_env)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "all", "--steps", str(steps), "--warmup", str(warmup),
           "--dump-outputs", dump_dir] + passthrough
    p = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True)
    if p.returncode != 0:
        sys.stderr.write(p.stdout[-4000:] + p.stderr[-4000:])
        raise SystemExit(f"bench.py failed ({p.returncode})")
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    return json.loads(lines[-1])


def write(path, out):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)


def load_dump(d):
    return {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith(".npy")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_sa_bench_3gbp_N1.json"))
    args, passthrough = ap.parse_known_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True).stdout.strip()
    runs, first_dump, dumps_equal = [], None, []
    out = {"gpu": gpu, "command": f"bench.py --gpus 1 --workload all --steps {args.steps} --warmup {args.warmup} " + " ".join(passthrough),
           "arms": {arm: env for arm, env in ARMS}, "order": "A B alternating, A = sa", "dumps": dumps_equal, "runs": runs}
    with tempfile.TemporaryDirectory() as tmp:
        for r in range(args.repeats):
            for arm, env in ARMS:
                d = os.path.join(tmp, f"{arm}_{r}")
                line = run_bench(env, args.steps, args.warmup, d, passthrough)
                dump = load_dump(d)
                if first_dump is None:
                    first_dump = dump
                same = dump.keys() == first_dump.keys() and all(np.array_equal(dump[k], first_dump[k]) for k in dump)
                dumps_equal.append({"arm": arm, "run": r, "arrays": len(dump), "equal_to_first_run": bool(same)})
                wl = {name: {"value": w["value"], "ms_per_step": w["ms_per_step"], "kernel_ms": w.get("kernel_ms"), "parity": w.get("parity")}
                      for name, w in line["workloads"].items()}
                runs.append({"arm": arm, "run": r, "value": line["value"], "index_tables": line["config"]["index_tables"],
                             "image_gb": line["config"]["image_gb"], "workloads": wl})
                print(f"{arm} run {r}: exact {line['value'] / 1e6:.1f} M q/s, dump equal: {same}", file=sys.stderr, flush=True)
                write(args.out, out)              # what is measured so far survives an interrupted run
    summary = {}
    for name in runs[0]["workloads"]:
        row = {}
        for arm, _ in ARMS:
            vals = [x["workloads"][name]["value"] for x in runs if x["arm"] == arm]
            ms = [x["workloads"][name]["ms_per_step"] for x in runs if x["arm"] == arm]
            km = [x["workloads"][name]["kernel_ms"] or {} for x in runs if x["arm"] == arm]
            row[arm] = {"value_median": statistics.median(vals), "value_spread": max(vals) - min(vals),
                        "ms_per_step_median": statistics.median(ms),
                        "search_ms_median": statistics.median([k.get("search", float("nan")) for k in km]),
                        "locate_ms_median": statistics.median([k.get("locate", float("nan")) for k in km]),
                        "parity_identical": all((x["workloads"][name]["parity"] or {}).get("identical", False) for x in runs if x["arm"] == arm)}
        row["value_ratio_sa_over_no_sa"] = row["sa"]["value_median"] / row["no_sa"]["value_median"]
        summary[name] = row
    out.update(summary=summary, all_dumps_equal=all(d["equal_to_first_run"] for d in dumps_equal))
    write(args.out, out)
    print(json.dumps({k: out[k] for k in ("gpu", "all_dumps_equal", "summary")}))


if __name__ == "__main__":
    main()
