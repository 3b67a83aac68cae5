#!/usr/bin/env python
"""bench.py -- throughput of the ScanFold scanning hot path on B200 (contract: see DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C2] [--dump-outputs DIR]

One "step" = one pass of the hot path over one record shard: for every window the native MFE fold
(+ structure), the partition function / ensemble diversity / centroid, r shuffles generated on the
device and their MFE folds, the z-score / p-value, and the ScanFold-Fold per-base-pair accumulation.
The workload is BASELINE.json configs[1] (C2): 29,903-nt synthetic SARS-CoV-2-like genome, 120-nt
window, step 1, 100 mono-nucleotide shuffles.  With N GPUs every rank scans its own contiguous range
of ~29.8 k windows of an N x 29,903-nt record (weak scaling).

`value`   windows/s with the record resident in HBM (sfb_scan_plan_run; CUDA events on the launch stream)
`e2e`     windows/s through the public host-buffer API scanfold_b200.scan.scan_record + fold accumulate
          (H2D of the record, D2H of every per-window result, host z/p, accumulate H2D/D2H) -- the headline
`--impl reference`  the reference's CPU path.  ViennaRNA is not installable here (no network, not in the
          image), so this arm times oracle/ (the CPU restatement of the same algorithms) on all host
          cores over a bounded sample of the same workload.
`--dump-outputs DIR`  after the timed steps, write what the last step of each arm computed as DIR/<name>.npy
          (float64, integers exact, 64 MB at most): scan_* = the ScanPlan.fetch() arrays of the device arm,
          e2e_* = the per-nucleotide results, window columns and partner table of the end-to-end arm.  Large
          per-window or per-entry arrays are a fixed, seeded sample (the indices are dumped beside them).  With
          several GPUs rank 0 writes: its own shard of the device arm and partner table, the gathered rest.
          The inputs are seeded, so two builds run with the same arguments can be compared file by file.
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

WORKLOADS = {
    # name: (L, W, step, r, shuffle, composition ACGU, seed)   -- SURVEY.md 8d
    "C1": (1000, 120, 1, 100, "mono", (0.25, 0.25, 0.25, 0.25), 1001),
    "C2": (29903, 120, 1, 100, "mono", (0.299, 0.184, 0.196, 0.321), 1002),
    # C2's geometry and composition on a record four genomes long: the fixed record of the 1/2/4/8-GPU strong-scaling
    # curve (a 29,903-nt record leaves 3.7 k windows = 0.25 s per GPU at N=8; 1 Mb (C4) is 66 s per step at N=1)
    "C2x4": (4 * 29903, 120, 1, 100, "mono", (0.299, 0.184, 0.196, 0.321), 1002),
}
# DRAM bytes per 120-nt fold of mfe3_kernel, from the ncu --set full capture named below (not measured in the run)
MFE3_DRAM_BYTES_PER_FOLD = 123.0
MFE3_TRAFFIC_SOURCE = ("dram__bytes_read.sum + dram__bytes_write.sum per fold from the ncu capture "
                       "profiles/r02y_mfe3_kernel_ncu.txt (24.8 MB per 202,000 folds), x folds per step")


def synth_record(name):
    L, W, step, r, stype, comp, seed = WORKLOADS[name]
    rng = np.random.Generator(np.random.PCG64(seed))
    idx = rng.choice(4, size=L, p=np.array(comp) / sum(comp))
    return "".join("ACGU"[k] for k in idx), W, step, r, stype


class ClockSampler:
    """SM clock, power and throttle reasons every 200 ms during the timed region (B200_PROFILING.md recipe).

    Read through NVML in a thread of this process: the recipe's `nvidia-smi --query-gpu=... -lms 200` loop was measured
    to slow the timed region by 3-10 % on some boxes (13.8 k / 14.8 k windows/s with it, 15.0 k / 15.3 k without, same
    box, r01r); the NVML calls return the same fields without that side effect.  nvidia-smi remains the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.samples = []      # (sm_mhz, sm_max_mhz, watts, reason bitmask)
        self.stop_flag = threading.Event()
        self.th = None
        self.source = None

    def start(self):
        if os.environ.get("SFB_NO_SAMPLER"):   # debugging only: measure the sampler's own perturbation
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            smax = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)

            def loop():
                while not self.stop_flag.is_set():
                    try:
                        self.samples.append((pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), smax,
                                             pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0, int(get_reasons(h))))
                    except pynvml.NVMLError:
                        pass
                    self.stop_flag.wait(0.2)

            self.th = threading.Thread(target=loop, daemon=True)
            self.th.start()
            self.source = "nvml"
            return
        except Exception:
            self.th = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
            self.source = "nvidia-smi"
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.source == "nvml":
            self.stop_flag.set()
            self.th.join(timeout=2)
            sm = [x[0] for x in self.samples]
            reasons = sorted(name for name, bit in self.REASONS if any(x[3] & bit for x in self.samples))
            return {"sm_mhz": float(np.median(sm)) if sm else None,
                    "sm_max_mhz": float(max(x[1] for x in self.samples)) if sm else None,
                    "power_w_max": max(x[2] for x in self.samples) if sm else None, "samples": len(sm),
                    "reasons": reasons, "source": "nvml, 200 ms period"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons),
                "source": "nvidia-smi -lms 200"}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_sample(seq, W, step, r, n_windows, rng_seed=7):
    """one bounded sample of the workload for the CPU arm: the first n_windows windows"""
    import random
    rnd = random.Random(rng_seed)
    natives = [seq[w * step:w * step + W] for w in range(n_windows)]
    folds = []
    for frag in natives:
        folds.append(frag)
        folds.extend("".join(rnd.sample(frag, W)) for _ in range(r))
    a = np.frombuffer("".join(folds).encode(), dtype=np.uint8).reshape(len(folds), W)
    n = np.frombuffer("".join(natives).encode(), dtype=np.uint8).reshape(len(natives), W)
    return a, n


def cpu_step(O, folds, natives, threads):
    """what the reference does per window on the CPU: r+1 MFE folds (ScanFoldFunctions.py:805-814), the
    native MFE with structure and one partition function with bpp / centroid / ED (ScanFold.py:494-504).
    The r+1 energy-only folds -- 99 % of the work -- go through the oracle's tuned batch path (reusable per-thread
    buffers, vectorised inner loops; tests check it equals the simple checker path fold by fold)."""
    t0 = time.perf_counter()
    O.fold_batch(folds, n_threads=threads, fast=True)
    t1 = time.perf_counter()
    O.fold_batch(natives, n_threads=threads)
    O.pf_batch(natives, n_threads=threads)
    return t1 - t0


def cpu_baseline_block(args, seq, W, step, r):
    from oracle import oracle as O
    O.lib()
    threads = host_threads()
    cw = args.cpu_windows
    folds, natives = cpu_sample(seq, W, step, r, cw)
    cpu_step(O, folds[:threads * 8], natives[:1], threads)     # page in, spin up
    t0 = time.perf_counter()
    t_folds = cpu_step(O, folds, natives, threads)
    dt = time.perf_counter() - t0
    return {"value": cw / dt, "unit": "windows/s", "cores": threads, "kind": "port",
            "ms_per_fold_per_core": t_folds * threads / len(folds) * 1e3,
            "sample": "first %d windows of %s, once (%d MFE folds + %d partition functions)"
                      % (cw, args.workload, len(folds) + cw, cw),
            "note": "oracle/ tuned batch path (gcc -O3 -march=native, %d threads); ViennaRNA itself is not installable here"
                    % threads}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    O.lib()
    seq, W, step, r, stype = synth_record(args.workload)
    threads = host_threads()
    nwin = args.cpu_windows
    folds, natives = cpu_sample(seq, W, step, r, nwin)
    for _ in range(max(args.warmup, 0) and 1):
        cpu_step(O, folds[:threads * (r + 1)], natives[:threads], threads)
    t0 = time.perf_counter()
    t_folds = 0.0
    for _ in range(args.steps):
        t_folds += cpu_step(O, folds, natives, threads)
    dt = time.perf_counter() - t0
    wps = nwin * args.steps / dt
    sample = "first %d windows of %s per step (%d MFE folds + %d native folds + %d partition functions)" % (
        nwin, args.workload, len(folds), nwin, nwin)
    line = {"impl": "reference", "metric": "windows/sec (MFE+%d shuffles+ED)" % r, "value": wps, "unit": "windows/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": workload_config(args.workload, 1),
            "cpu_baseline": {"value": wps, "unit": "windows/s", "cores": threads, "kind": "port", "sample": sample,
                             "ms_per_fold_per_core": t_folds * threads / (len(folds) * args.steps) * 1e3,
                             "note": "ViennaRNA (the reference's fold engine) is not installable offline; "
                                     "oracle/ is the CPU restatement of the same algorithms, tuned batch path "
                                     "(gcc -O3 -march=native, reusable per-thread buffers, vectorised inner loops)"},
            "e2e": {"value": wps, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(name, n_gpus):
    L, W, step, r, stype, comp, seed = WORKLOADS[name]
    return {"workload": "%s: one %d-nt synthetic record (the same record for every N), window %d, step %d, %d %s "
                        "shuffles, PF/ED on; `value` times the scan kernels (shuffles, MFE folds, partition function), "
                        "`e2e` adds host buffers, z/p and the ScanFold-Fold accumulation kernels" % (name, L, W, step, r, stype),
            "record_nt": L, "window": W, "step": step, "shuffles": r, "shuffle_type": stype,
            "seed": seed, "l2": "flushed between steps (256 MiB write)",
            "parallelism": "windows of the one record sharded by range over %d GPU(s); accumulator halo rows over NCCL "
                           "send/recv; every rank aggregates the nucleotides it owns, rank 0 gathers the per-nucleotide "
                           "results and the window columns" % n_gpus}


def result_sha(agg, table_digest, table):
    """Digest of what a run produces before the writers: the per-nucleotide ScanFold-Fold results (best partner and its
    metrics), an order-independent checksum of the merged partner table, and the per-window columns.
    Identical for every N (integer / exact-sum accumulators, shuffles keyed by absolute window index)."""
    import hashlib
    h = hashlib.sha256()
    h.update(np.uint64(table_digest).tobytes())
    for a, dt in ((agg.coord, np.int64), (agg.part, np.int64), (agg.cov_z, np.float64), (agg.mean_z, np.float64),
                  (agg.mean_mfe, np.float64), (agg.mean_ed, np.float64), (agg.total_windows, np.int64), (agg.num_bp, np.int64)):
        h.update(np.ascontiguousarray(a, dtype=dt).tobytes())
    for a, dt in ((table.mfe_dcal, np.int64), (table.native_unconstrained_dcal, np.int64), (table.z, np.float64),
                  (table.p, np.float64), (table.ed, np.float64), (table.pair_tbl, np.int16), (table.centroid_tbl, np.int16)):
        h.update(np.ascontiguousarray(a, dtype=dt).tobytes())
    return h.hexdigest()[:16]


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE_WINDOWS = 4096      # rows of the [n, r] shuffle energies and [n, W] structures
DUMP_SAMPLE_ENTRIES = 65536     # entries of the partner table
NT_RESULT_FIELDS = ("coord", "part", "cov_z", "mean_z", "mean_mfe", "mean_ed", "total_windows", "num_bp")


def sample_indices(n, k, seed):
    """sorted indices of a fixed, seeded sample of k out of n (all n when n <= k)"""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))


def scan_outputs(res):
    """ScanPlan.fetch() of the device arm: per-window columns in full, the wide arrays for a sample of windows"""
    out = {"scan_" + k: getattr(res, k) for k in ("mfe_dcal", "native_unconstrained_dcal", "ed", "ensemble_dG")}
    rows = sample_indices(res.n, DUMP_SAMPLE_WINDOWS, 1)
    out["scan_sample_windows"] = rows
    for k in ("shuffle_dcal", "pair_tbl", "centroid_tbl"):
        out["scan_" + k] = getattr(res, k)[rows]
    return out


def e2e_outputs(agg, wtable, ptable):
    """the end-to-end arm: per-nucleotide results, per-window columns, the partner table for a sample of entries"""
    out = {"e2e_nt_" + k: getattr(agg, k) for k in NT_RESULT_FIELDS}
    for k in ("mfe", "z", "p", "ed"):
        out["e2e_window_" + k] = getattr(wtable, k)
    if wtable.final is not None:
        out["e2e_final_window_mfe_z_p_ed"] = [wtable.final[k] for k in ("mfe", "z", "p", "ed")]
    out["e2e_partner_nt_ptr"] = ptable.nt_ptr
    out["e2e_partner_coord"] = ptable.coord
    entries = sample_indices(len(ptable.partner), DUMP_SAMPLE_ENTRIES, 2)
    out["e2e_partner_sample_entries"] = entries
    for k in ("partner", "count", "first_seen"):
        out["e2e_partner_" + k] = getattr(ptable, k)[entries]
    out["e2e_partner_sums"] = ptable.sums[:, entries]
    return out


def write_outputs(path, arrays):
    """every array as <path>/<name>.npy in float64 (exact for the integer arrays: all below 2^53)"""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes, more than %d" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from scanfold_b200 import engine, foldstep, multigpu, pipeline, scan, workcount

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    engine.init(local)
    stream = torch.cuda.current_stream()
    engine.set_stream(stream.cuda_stream)

    seq, W, step, r, stype = synth_record(args.workload)      # ONE record whatever N: strong scaling
    L = len(seq)
    total = scan.n_windows_of(L, W, step)
    if args.windows:
        total = min(total, args.windows)
    w0, w1 = multigpu.shard_windows(total, world, rank)
    nwin = w1 - w0
    final = (w1 == scan.n_windows_of(L, W, step))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident arm: `value`
    plan = engine.ScanPlan(seq, W, step, r, shuffle_type=stype, seed=42, first_window=w0, n_windows=nwin,
                           final_window=final, want_pf=True)
    for _ in range(args.warmup):
        plan.run()
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms_mfe = ms_pf = 0.0
    launches = 0
    ev0.record(stream)
    for _ in range(args.steps):
        flush.zero_()
        plan.run()
        ms_mfe += plan.ms_mfe
        ms_pf += plan.stage_ms["pf"]
        launches += plan.n_launches
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms_dev = ev0.elapsed_time(ev1)
    dump = scan_outputs(plan.fetch()) if args.dump_outputs and rank == 0 else None
    plan.close()

    # ---------------- end-to-end arm through the public API with host buffers: `e2e`
    trace = os.environ.get("SFB_BENCH_TRACE")
    grp = dist if world > 1 else None

    def e2e_step():
        tt = [time.perf_counter()]
        t = scan.scan_record(seq, W, step, r, shuffle_type=stype, seed=42, first_window=w0, n_windows=nwin,
                             final_window=final)
        tt.append(time.perf_counter())
        z100, mfe100, ed100 = pipeline.fold_inputs(t)
        acc = engine.Accumulator(L, W, step, w0, t.pair_tbl, z100, mfe100, ed100)
        try:        # halo rows go to their owners over NCCL; every rank keeps the nucleotides it owns
            ptable = multigpu.own_partner_table(acc, W, step, rank, world, grp, total)
            launches_e2e[0] = acc.n_launches
        finally:
            acc.close()
        tt.append(time.perf_counter())
        # ScanFold.py:1051-1260 on the owned nucleotides; rank 0 gathers the per-nucleotide results and the window columns
        agg, _, _ = multigpu.aggregate_distributed(ptable, seq, rank, world, grp)
        wtable = multigpu.gather_window_tables(t, rank, world, grp)
        tt.append(time.perf_counter())
        if trace and rank == 0:
            sys.stderr.write("e2e step: scan_record %.1f ms (device %.1f), accumulate %.1f ms, aggregate + gather %.1f ms\n" % (
                (tt[1] - tt[0]) * 1e3, t.ms_total, (tt[2] - tt[1]) * 1e3, (tt[3] - tt[2]) * 1e3))
        return t, ptable, agg, wtable, [b - a for a, b in zip(tt, tt[1:])]

    launches_e2e = [0]
    e2e_steps = args.e2e_steps or args.steps
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    parts = np.zeros(3)
    for _ in range(e2e_steps):
        flush.zero_()
        t, own_table, agg, wtable, dts = e2e_step()
        parts += dts
    barrier()
    ms_e2e = (time.perf_counter() - t0) * 1e3
    table_digest = multigpu.table_checksum(own_table, rank, world, grp)      # outside the timed region
    n_slots = nwin + (1 if final else 0)
    h2d = L + nwin * W * 2 + nwin * 12
    d2h = n_slots * (4 + 4 + 4 * r + 2 * W + 2 * W + 8 + 8) + len(own_table.partner) * 60 + own_table.n_nt * 4

    # ---------------- max over ranks
    tt = torch.tensor([ms_dev, ms_e2e, ms_mfe, ms_pf], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([float(nwin), float(launches), float(h2d), float(d2h)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    ms_dev, ms_e2e, ms_mfe_max, ms_pf_max = tt.tolist()
    total_windows, total_launches, h2d_all, d2h_all = cnt.tolist()

    if rank == 0:
        if dump is not None:
            dump.update(e2e_outputs(agg, wtable, own_table))
            write_outputs(args.dump_outputs, dump)
        folds_per_window = r + 1
        n_folds = (nwin + (1 if final else 0)) * folds_per_window
        cells = workcount.cells(W)
        dense = workcount.dense_relaxations(W)
        rs = np.random.default_rng(5)
        sample_w = rs.integers(0, L - W, size=24)
        useful_nat = [workcount.useful_relaxations(seq[s:s + W]) for s in sample_w[:12]]
        useful = float(np.mean(useful_nat + [workcount.useful_relaxations("".join(rs.permutation(list(seq[s:s + W]))))
                                             for s in sample_w[12:]]))
        peak_addmin = engine.microbench(0)
        peak_lds = engine.microbench(1)
        peak_dfma = engine.microbench(2)
        mfe_s = ms_mfe / args.steps * 1e-3          # MFE kernels of one step on this rank (library CUDA events)
        pf_s = ms_pf / args.steps * 1e-3            # partition-function kernels of one step on this rank
        achieved = useful * n_folds / mfe_s
        pf_fma = 2.0 * float(np.mean(useful_nat))   # SURVEY 8d: one FMA per relaxation, inside + outside
        value = total_windows * args.steps / (ms_dev * 1e-3)
        e2e = total_windows * e2e_steps / (ms_e2e * 1e-3)
        line = {
            "metric": "windows/sec (MFE+%d shuffles+ED)" % r, "value": value, "unit": "windows/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": workload_config(args.workload, world),
            "folds_per_s": value * folds_per_window, "dp_cells_per_s": value * folds_per_window * cells,
            "result_sha": result_sha(agg, table_digest, wtable),
            "e2e": {"value": e2e, "unit": "windows/s", "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
                    "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps,
                    "rank0_ms_per_step": {"scan_record": parts[0] / e2e_steps * 1e3,
                                          "accumulate_halo_compact": parts[1] / e2e_steps * 1e3,
                                          "aggregate_and_gather_to_rank0": parts[2] / e2e_steps * 1e3}},
            "gpu_launches": int(total_launches), "gpu_launches_e2e_per_step": int(t.n_launches + launches_e2e[0]),
            "roofline": {"bound": "int_alu", "kernel": "mfe3_kernel (+ int32 redo of flagged folds)", "achieved": achieved / 1e9,
                         "peak": peak_addmin / 1e9, "unit": "G add-min/s", "frac": achieved / peak_addmin,
                         "peak_source": "sfb_microbench VIADDMNMX rate measured in this run (MEASURED_PEAKS.json "
                                        "has no integer peak; HBM is not the bound)",
                         "algorithmic_ops_per_fold": useful, "dense_ops_per_fold": dense,
                         "achieved_dense": dense * n_folds / mfe_s / 1e9,
                         "smem_ld32_peak_per_s": peak_lds, "kernel_ms_per_step": mfe_s * 1e3,
                         "kernel_share_of_step": ms_mfe / ms_dev,
                         "hbm_algorithmic_bytes_per_fold": W + 4,
                         "traffic": (MFE3_DRAM_BYTES_PER_FOLD * n_folds) if W == 120 else None,
                         "traffic_source": MFE3_TRAFFIC_SOURCE},
            "roofline_pf": {"bound": "fp64_fma", "kernel": "pf2_kernel", "achieved": pf_fma * nwin / pf_s / 1e9,
                            "peak": peak_dfma / 1e9, "unit": "G fp64 FMA/s", "frac": pf_fma * nwin / pf_s / peak_dfma,
                            "peak_source": "sfb_microbench DFMA rate measured in this run",
                            "algorithmic_fma_per_window": pf_fma, "kernel_ms_per_step": pf_s * 1e3,
                            "kernel_share_of_step": ms_pf / ms_dev, "windows_per_s": nwin / pf_s},
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_block(args, seq, W, step, r)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2x4", choices=sorted(WORKLOADS))
    ap.add_argument("--windows", type=int, default=0, help="debug: cap the windows of the record")
    ap.add_argument("--e2e-steps", type=int, default=0, help="end-to-end steps (default: --steps)")
    ap.add_argument("--cpu-windows", type=int, default=192, help="windows per CPU sample step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of each arm as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
