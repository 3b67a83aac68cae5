"""Window-averaged base-pair probabilities on the GPU (sfb_pairprob_*, --pair_probs): the device table, reduced on the
device, against the restatement of the definition from per-window oracle partition functions (|dP|, |dpaired| <= 1e-9,
the bpp tolerance of the PF tests); windows out of the fp64 range counted once; bit-identical int64 sums however the
scan is split; and the CLI files."""
import os
import random
import shutil
import subprocess
import sys

import numpy as np
import pytest

import param_tables as PT
from pairprob_ref import CUTOFF, pair_list, restate, window_bpp
from test_gpu_param_edges import loaded
from test_host_pipeline import GOLDEN, load_case
from util import rand_seqs

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def device_table(engine, seq, W, step, r=2, first_window=0, n_windows=None, **kw):
    from scanfold_b200 import scan
    n = (len(seq) - W) // step + 1 - first_window if n_windows is None else n_windows
    t = engine.PairProbTable(len(seq), W, step, first_window, n)
    scan.scan_record(seq, W, step, r, seed=4, first_window=first_window, n_windows=n, pairprob=t, **kw)
    return t


def check_rows(t, seq, W, step, wa, wb, row_lo, row_hi, hc=None, max_span=0, temperature=37.0):
    """rows [row_lo, row_hi) of the device table (record coordinates) against the restatement over windows [wa, wb),
    which must hold every window that holds those rows"""
    bpps = [window_bpp(seq, W, step, w, hc=hc, max_span=max_span, temperature=temperature) for w in range(wa, wb)]
    a = wa * step
    sub_L = (wb - 1 - wa) * step + W
    paired, n_i, P, _ = restate(sub_L, W, step, bpps)
    dp, di, dj, dprob = t.reduce(row_lo - t.nt0, row_hi - row_lo)
    assert np.max(np.abs(dp - paired[row_lo - a:row_hi - a])) <= 1e-9
    Pr = np.zeros_like(P)
    Pr[row_lo - a:row_hi - a] = P[row_lo - a:row_hi - a]
    ri, rj, rp = pair_list(Pr)
    ref = {(x + a, y + a): v for x, y, v in zip(ri.tolist(), rj.tolist(), rp.tolist())}
    got = {(x, y): v for x, y, v in zip(di.tolist(), dj.tolist(), dprob.tolist())}
    assert list(got) == sorted(got)                       # row order, then column order
    for key in set(ref) | set(got):
        v = ref.get(key, P[key[0] - 1 - a, key[1] - 1 - a])
        if abs(v - CUTOFF) > 1e-9:
            assert key in got and key in ref, key
            assert abs(got[key] - v) <= 1e-9, (key, got[key], v)
    return len(got)


def check_record(engine, seq, W, step, hc=None, max_span=0, temperature=37.0, **kw):
    n = (len(seq) - W) // step + 1
    t = device_table(engine, seq, W, step, hc=hc, max_span=max_span, temperature=temperature, **kw)
    try:
        return check_rows(t, seq, W, step, 0, n, 0, (n - 1) * step + W, hc=hc, max_span=max_span, temperature=temperature)
    finally:
        t.close()


@pytest.mark.parametrize("W,step,L", [(40, 1, 100), (120, 1, 150), (120, 7, 270), (121, 7, 250), (200, 7, 260)])
def test_matches_restatement(engine, oracle, W, step, L):
    """W <= 120: pf2 (shared-memory kernel); 121 and 200: pf.cu"""
    seq = rand_seqs(W * 1000 + step, 1, L)[0]
    assert check_record(engine, seq, W, step) > 0


def test_flag_constraints_pf2_and_brackets_pf(engine, oracle):
    rng = random.Random(7)
    seq = rand_seqs(71, 1, 150)[0]
    flags = "".join(rng.choice("......x<>") for _ in seq)
    check_record(engine, seq, 60, 3, hc=flags)
    hc = list("." * len(seq))
    for i, j in ((10, 40), (12, 38), (70, 120), (95, 110)):
        hc[i], hc[j] = "(", ")"
    hc[50] = "x"
    check_record(engine, seq, 60, 3, hc="".join(hc))


def test_react_leaves_the_pf_unconstrained(engine, oracle):
    seq = rand_seqs(72, 1, 140)[0]
    react = np.concatenate([[-999.0], np.clip(np.random.default_rng(1).exponential(0.5, len(seq)), 0, 4)])
    check_record(engine, seq, 60, 3, react=react)


def test_span_and_temperature(engine, oracle):
    seq = rand_seqs(73, 1, 160)[0]
    check_record(engine, seq, 80, 5, max_span=50)
    try:
        check_record(engine, seq, 60, 7, temperature=25.0)
    finally:
        oracle.set_temperature(37.0)


def test_step_greater_than_window(engine, oracle):
    seq = rand_seqs(74, 1, 200)[0]
    W, step = 40, 55
    n = (len(seq) - W) // step + 1
    t = device_table(engine, seq, W, step)
    try:
        check_rows(t, seq, W, step, 0, n, 0, (n - 1) * step + W)
        paired = t.reduce()[0]
        assert np.all(paired[W:step] == 0) and np.all(t.rows()[W:step] == 0)
    finally:
        t.close()


def test_windows_straddling_a_plan_chunk(engine, oracle):
    """more than 65,536 windows: the plan runs in chunks; the rows around the boundary equal the restatement"""
    rng = np.random.default_rng(21)
    W = 40
    L = 65536 + 300 + W - 1
    seq = "".join("ACGU"[k] for k in rng.integers(0, 4, L))
    t = engine.PairProbTable(L, W, 1, 0, L - W + 1)
    try:
        engine.scan(seq, W, 1, 2, seed=3, pairprob=t)     # one plan (scan_record would split it into parts)
        check_rows(t, seq, W, 1, 65536 - 70, 65536 + 50, 65536 - 25, 65536 + 10)
    finally:
        t.close()


def test_out_of_range_windows_are_counted_once(engine, oracle, tmp_path):
    """windows whose Z leaves the fp64 range under the default scale (a GC repeat of 400 nt at 37 C on pf.cu; stack x 3
    at 120 nt on pf2) add the probabilities of their rescaled retry, once"""
    seq = rand_seqs(17, 1, 200)[0] + "GGGGGCCCCC" * 40 + rand_seqs(18, 1, 200)[0]
    with pytest.raises(RuntimeError):
        oracle.pf(seq[200:600], pf_scale=0)              # the default scale overflows: the scan takes the retry
    check_record(engine, seq, 400, 100)
    with loaded(engine, oracle, PT.stack_scaled(3), tmp_path):
        seq = "GGGGGCCCCC" * 12 + rand_seqs(3, 1, 40)[0] + "GC" * 60
        with pytest.raises(RuntimeError):
            oracle.pf(seq[:120], pf_scale=0)
        check_record(engine, seq, 120, 20)


def test_split_scans_are_bit_identical(engine, oracle, monkeypatch):
    from scanfold_b200 import scan
    seq = rand_seqs(75, 1, 400)[0]
    W, step = 60, 3
    whole = device_table(engine, seq, W, step)
    ref = whole.rows()
    whole.close()
    for parts in (7, 16, 40):
        monkeypatch.setattr(scan, "PIPELINE_WINDOWS", parts)
        t = device_table(engine, seq, W, step)
        assert np.array_equal(t.rows(), ref), parts
        t.close()
    # two shards of the same record into one table, and the halo merge of two shard tables, give the same sums
    n = (len(seq) - W) // step + 1
    t = engine.PairProbTable(len(seq), W, step, 0, n)
    scan.scan_record(seq, W, step, 2, seed=4, first_window=0, n_windows=30, pairprob=t)
    scan.scan_record(seq, W, step, 2, seed=4, first_window=30, n_windows=n - 30, pairprob=t)
    assert np.array_equal(t.rows(), ref)
    t.close()
    a = device_table(engine, seq, W, step, first_window=0, n_windows=30)
    b = device_table(engine, seq, W, step, first_window=30, n_windows=n - 30)
    halo = a.n_nt - b.nt0
    b.merge_tensors(0, halo, *a.export_tensors(b.nt0, halo))
    assert np.array_equal(np.concatenate([a.rows(0, b.nt0), b.rows()]), ref)
    a.close()
    b.close()


def test_argument_errors(engine):
    from scanfold_b200 import engine as E
    t = E.PairProbTable(200, 40, 2, 10, 20)
    try:
        for kw, msg in ((dict(first_window=0, n_windows=5), "range"), (dict(first_window=25, n_windows=10), "range"),
                        (dict(want_pf=False), "want_pf")):
            kw = dict(dict(first_window=10, n_windows=20, final_window=False), **kw)
            with pytest.raises(E.EngineError, match=msg):
                E.ScanPlan("A" * 200, 40, 2, 1, pairprob=t, **kw)
        with pytest.raises(E.EngineError, match="window or step"):
            E.ScanPlan("A" * 200, 40, 1, 1, first_window=10, n_windows=20, final_window=False, pairprob=t)
        with pytest.raises(E.EngineError, match="row range"):
            t.reduce(0, t.n_nt + 1)
    finally:
        t.close()
    with pytest.raises(E.EngineError):
        E.PairProbTable(200, 40, 2, 0, 100)


def _parse_outputs(folder, outname):
    wig = open(os.path.join(folder, outname + ".pairprob.wig")).read().split("\n")
    assert wig[0] == "variableStep chrom=UserInput span=1"
    pos, paired = zip(*[(int(a), float(b)) for a, b in (ln.split("\t") for ln in wig[1:] if ln)])
    txt = open(os.path.join(folder, outname + ".pairprob.txt")).read().split("\n")
    assert txt[0] == "i\tj\tprobability"
    pairs = {(int(a), int(b)): float(c) for a, b, c in (ln.split("\t") for ln in txt[1:] if ln)}
    bp = open(os.path.join(folder, "IGV_BP_Track." + outname + ".pairprob.bp")).read().split("\n")
    assert all(ln.startswith("color:\t") for ln in bp[:4])
    arcs = {}
    for ln in bp[4:]:
        if ln:
            name, i, i2, j, j2, c = ln.split("\t")
            assert name == "UserInput" and i == i2 and j == j2
            arcs[(int(i), int(j))] = int(c)
    return np.array(pos), np.array(paired), pairs, arcs


@pytest.mark.parametrize("name", ["mono_w40", "hc_w40"])
def test_cli_pair_probs(name, tmp_path, monkeypatch, engine, oracle):
    from scanfold_b200 import cli
    d = os.path.join(GOLDEN, name)
    case = load_case(name)
    for f in ("input.fa", "constraints.dbn", "trace.npz"):
        if os.path.exists(os.path.join(d, f)):
            shutil.copy(os.path.join(d, f), tmp_path / f)
    args = [a if a != "constraints.dbn" else str(tmp_path / "constraints.dbn") for a in case["args"]]
    monkeypatch.chdir(tmp_path)
    cli.main(["input.fa"] + args + ["--parity_shuffles", "trace.npz", "--pair_probs"])
    out = tmp_path / case["record"]
    exp_dir = os.path.join(d, "expected")
    exp = sorted(os.listdir(exp_dir))
    outname = "%s.win_%d.stp_%d.rnd_%d.shfl_mono" % (case["record"], case["W"], case["step"], case["r"])
    new = [outname + ".pairprob.wig", outname + ".pairprob.txt", "IGV_BP_Track." + outname + ".pairprob.bp"]
    assert sorted(os.listdir(out)) == sorted(exp + new)
    for f in exp:
        assert open(out / f).read() == open(os.path.join(exp_dir, f)).read(), f
    hc = open(tmp_path / "constraints.dbn").readlines()[2].rstrip("\n") if "--constraints" in args else None
    seq, W, step = case["seq"].upper(), case["W"], case["step"]
    n = (len(seq) - W) // step + 1
    paired, n_i, P, _ = restate(len(seq), W, step, [window_bpp(seq, W, step, w, hc=hc) for w in range(n)])
    pos, dpaired, pairs, arcs = _parse_outputs(str(out), outname)
    assert np.array_equal(pos, np.nonzero(n_i)[0] + 1)
    assert np.max(np.abs(dpaired - paired[pos - 1])) <= 1e-6
    ri, rj, rp = pair_list(P)
    for i, j, v in zip(ri.tolist(), rj.tolist(), rp.tolist()):
        if v >= CUTOFF + 1e-6:
            assert abs(pairs[(i, j)] - v) <= 1e-6
    for (i, j), v in pairs.items():
        assert abs(P[i - 1, j - 1] - v) <= 1e-6
        assert ((i, j) in arcs) == (P[i - 1, j - 1] >= 0.1) or abs(P[i - 1, j - 1] - 0.1) < 1e-9
    for (i, j), c in arcs.items():
        assert c == int(np.searchsorted([0.1, 0.3, 0.5, 0.8], P[i - 1, j - 1], side="right")) - 1
    # without the flag the folder holds exactly the golden file set
    monkeypatch.chdir(tmp_path)
    cli.main(["input.fa"] + args + ["--parity_shuffles", "trace.npz", "--out_name", "noflag"])
    assert sorted(os.listdir(tmp_path / "noflag")) == exp


def test_cli_two_gpus_write_the_same_files(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs (found %d)" % torch.cuda.device_count())
    d = os.path.join(GOLDEN, "step7_w40")
    shutil.copy(os.path.join(d, "input.fa"), tmp_path / "input.fa")
    base = ["input.fa", "-w", "40", "-r", "10", "-s", "7", "--pair_probs"]
    env = dict(os.environ, PYTHONPATH=ROOT)
    runs = {"one": [sys.executable, "-m", "scanfold_b200.cli"],
            "two": [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                    "--master-addr", "127.0.0.1", "--master-port", str(29700 + os.getpid() % 200), "-m",
                    "scanfold_b200.cli"]}
    for name, cmd in runs.items():
        p = subprocess.run(cmd + base + ["--out_name", name], cwd=tmp_path, env=env, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=600)
        assert p.returncode == 0, p.stdout[-3000:]
    files = [f for f in os.listdir(tmp_path / "one") if "pairprob" in f]
    assert len(files) == 3
    for f in files:
        assert (tmp_path / "one" / f).read_bytes() == (tmp_path / "two" / f).read_bytes(), f
