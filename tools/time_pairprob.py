"""Cost of --pair_probs on the C2 geometry (120 nt, step 1, 100 shuffles): the 29,903-nt record (C2) and the 119,612-nt
bench record (C2x4).  Per workload, alternating runs without and with a pair-probability table attached:
  device  one ScanPlan over all windows: CUDA-event time of the PF stage (stage_ms["pf"]) and of the whole run
  e2e     scan.scan_record (pipelined parts, fetch, z / p statistics; with the table also its creation and reduce())
          on the host clock -> windows/s
  table   PairProbTable creation, reduce() of every row (count + scan + emit kernels, copies) on the host clock
Prints the card name and power limit read in the same process, then one JSON line.
usage: python tools/time_pairprob.py [--workloads C2,C2x4] [--reps 3]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import bench  # noqa: E402
from scanfold_b200 import engine, scan  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip().split("\n")[0]
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="C2,C2x4")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    engine.init(0)
    out = {"card": card(), "workloads": {}}
    print("card:", out["card"])
    for name in a.workloads.split(","):
        seq, W, step, r, stype = bench.synth_record(name)
        L = len(seq)
        n = scan.n_windows_of(L, W, step)
        rec = {k: [] for k in ("pf_ms_off", "pf_ms_on", "run_ms_off", "run_ms_on", "e2e_s_off", "e2e_s_on",
                               "table_begin_ms", "reduce_ms", "n_pairs")}
        plan = engine.ScanPlan(seq, W, step, r, shuffle_type=stype, seed=42)
        plan.run()                                            # warm-up: module load, scratch, both PF specialisations
        t = engine.PairProbTable(L, W, step, 0, n)
        p2 = engine.ScanPlan(seq, W, step, r, shuffle_type=stype, seed=42, pairprob=t)
        p2.run()
        p2.close()
        t.reduce()
        t.close()
        for rep in range(a.reps):
            plan.run()
            rec["pf_ms_off"].append(plan.stage_ms["pf"])
            rec["run_ms_off"].append(plan.ms_total)
            t0 = time.perf_counter()
            t = engine.PairProbTable(L, W, step, 0, n)
            rec["table_begin_ms"].append((time.perf_counter() - t0) * 1e3)
            p2 = engine.ScanPlan(seq, W, step, r, shuffle_type=stype, seed=42, pairprob=t)
            p2.run()
            rec["pf_ms_on"].append(p2.stage_ms["pf"])
            rec["run_ms_on"].append(p2.ms_total)
            p2.close()
            t0 = time.perf_counter()
            res = t.reduce()
            rec["reduce_ms"].append((time.perf_counter() - t0) * 1e3)
            rec["n_pairs"].append(len(res[1]))
            t.close()
            t0 = time.perf_counter()
            scan.scan_record(seq, W, step, r, shuffle_type=stype, seed=42)
            rec["e2e_s_off"].append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            t = engine.PairProbTable(L, W, step, 0, n)
            scan.scan_record(seq, W, step, r, shuffle_type=stype, seed=42, pairprob=t)
            t.reduce()
            t.close()
            rec["e2e_s_on"].append(time.perf_counter() - t0)
        plan.close()
        med = {k: float(np.median(v)) for k, v in rec.items()}
        spread = {k: [float(min(v)), float(max(v))] for k, v in rec.items()}
        med["e2e_windows_per_s_off"] = n / med["e2e_s_off"]
        med["e2e_windows_per_s_on"] = n / med["e2e_s_on"]
        out["workloads"][name] = {"L": L, "W": W, "step": step, "r": r, "n_windows": n, "median": med, "min_max": spread}
        print("%s: %d windows  PF stage %.1f -> %.1f ms (+%.1f%%)  plan run %.1f -> %.1f ms (+%.1f%%)" % (
            name, n, med["pf_ms_off"], med["pf_ms_on"], 100 * (med["pf_ms_on"] / med["pf_ms_off"] - 1), med["run_ms_off"],
            med["run_ms_on"], 100 * (med["run_ms_on"] / med["run_ms_off"] - 1)))
        print("%s: scan_record %.0f -> %.0f windows/s (%.1f%%)  table begin %.1f ms  reduce+fetch %.1f ms  %d pairs" % (
            name, med["e2e_windows_per_s_off"], med["e2e_windows_per_s_on"],
            100 * (med["e2e_windows_per_s_on"] / med["e2e_windows_per_s_off"] - 1), med["table_begin_ms"],
            med["reduce_ms"], med["n_pairs"]))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
