"""Window-averaged base-pair probabilities (--pair_probs) on the CPU: the window counts of the definition, the
exclusion of the final-window slot, the three file formats, and the multi-rank reduction (gloo, NumPy stand-in of the
device table) against one rank."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from pairprob_ref import NumpyPairProbTable, pair_list, restate, window_bpp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def brute_counts(L, W, step):
    n = (L - W) // step + 1
    n_i = np.zeros(L, dtype=np.int64)
    n_ij = np.zeros((L, L), dtype=np.int64)
    for w in range(n):
        n_i[w * step:w * step + W] += 1
        n_ij[w * step:w * step + W, w * step:w * step + W] += 1
    return n, n_i, n_ij


@pytest.mark.parametrize("L,W,step", [(90, 30, 1), (131, 40, 7), (140, 20, 25), (60, 60, 1), (200, 120, 13)])
def test_window_counts(L, W, step):
    from scanfold_b200.engine import windows_holding
    n, n_i, n_ij = brute_counts(L, W, step)
    k = np.arange(L)
    assert np.array_equal(windows_holding(k, k, W, step, n), n_i)
    i, j = np.triu_indices(L)
    assert np.array_equal(windows_holding(i, j, W, step, n), n_ij[i, j])
    if step > W:
        assert (n_i == 0).any()       # gaps between windows: no window holds those nucleotides


def test_final_slot_is_not_a_window():
    """the last regular window of 107 nt / W 40 / step 7 ends at 103: the final-window slot [67, 107) adds nothing"""
    seq = "GGGAAACCCAGCUAGCUAGGCAUCGAUCGGAUCCGAUGCUAGCUAGCGGAUCCGAUCGAUGCUAGCGCGAUAUAUCGCGGCCAUUAGGCCUAAGCUUAGCGCGCUAAUU"[:107]
    L, W, step = len(seq), 40, 7
    n = (L - W) // step + 1
    bpps = [window_bpp(seq, W, step, w) for w in range(n)]
    paired, n_i, P, N = restate(L, W, step, bpps)
    assert (n - 1) * step + W == 103
    assert np.all(n_i[103:] == 0) and np.all(paired[103:] == 0) and np.all(P[:, 103:] == 0)
    # and it is the average the definition asks for
    for i, j in [(70, 95), (64, 100), (10, 40)]:
        terms = [bpps[w][i - w * step, j - w * step] for w in range(n) if w * step <= i and j < w * step + W]
        assert N[i, j] == len(terms)
        assert P[i, j] == pytest.approx(sum(terms) / len(terms) if terms else 0.0, abs=1e-15)
    # the stand-in table reduces to the same values
    t = NumpyPairProbTable(L, W, step, 0, n)
    for w, B in enumerate(bpps):
        t.add_window(w, B)
    pd, ii, jj, pp = t.reduce()
    assert len(pd) == 103
    assert np.max(np.abs(pd - paired[:103])) <= 1e-9
    ri, rj, rp = pair_list(P)
    far = np.abs(rp - 0.01) > 1e-9
    got = {(a, b): c for a, b, c in zip(ii.tolist(), jj.tolist(), pp.tolist())}
    for a, b, c in zip(ri[far].tolist(), rj[far].tolist(), rp[far].tolist()):
        assert abs(got[(a, b)] - c) <= 1e-9


def test_file_formats(tmp_path):
    from scanfold_b200 import writers
    paired = np.array([0.5, 0.25, 0.0, 0.125])
    covered = np.array([True, True, False, True])
    writers.write_pairprob_wig(str(tmp_path / "a.wig"), paired, covered, "chr")
    assert (tmp_path / "a.wig").read_text() == "variableStep chrom=chr span=1\n1\t0.500000\n2\t0.250000\n4\t0.125000\n"
    i = np.array([1, 1, 2, 3, 5], dtype=np.int32)
    j = np.array([9, 12, 8, 30, 7], dtype=np.int32)
    p = np.array([0.01, 0.1, 0.3, 0.8, 0.79999999])
    writers.write_pairprob_txt(str(tmp_path / "a.txt"), i, j, p)
    assert (tmp_path / "a.txt").read_text() == (
        "i\tj\tprobability\n1\t9\t0.010000\n1\t12\t0.100000\n2\t8\t0.300000\n3\t30\t0.800000\n5\t7\t0.800000\n")
    writers.write_pairprob_bp(str(tmp_path / "a.bp"), i, j, p, "chr")
    assert (tmp_path / "a.bp").read_text() == (
        "color:\t199\t199\t199\t0.1 to 0.3\ncolor:\t236\t236\t136\t0.3 to 0.5\n"
        "color:\t89\t222\t111\t0.5 to 0.8\ncolor:\t55\t129\t255\t0.8 to 1\n"
        "chr\t1\t1\t12\t12\t0\nchr\t2\t2\t8\t8\t1\nchr\t3\t3\t30\t30\t3\nchr\t5\t5\t7\t7\t2\n")


WORKER = textwrap.dedent("""
    import os, sys
    import numpy as np
    import torch.distributed as dist
    sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
    from pairprob_ref import NumpyPairProbTable, CUTOFF
    from scanfold_b200 import multigpu
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    L, W, step = %(L)d, %(W)d, %(step)d
    n = (L - W) // step + 1
    rng = np.random.default_rng(5)
    bpps = []
    for w in range(n):           # synthetic per-window probabilities: sparse, some above and some below the cutoff
        B = np.triu(rng.random((W, W)) ** 6, 4) * (rng.random((W, W)) < 0.3)
        bpps.append(B / max(1.0, (B.sum(0) + B.sum(1)).max()))
    def table(w0, w1):
        t = NumpyPairProbTable(L, W, step, w0, w1 - w0)
        for w in range(w0, w1):
            t.add_window(w, bpps[w])
        return t
    w0, w1 = multigpu.shard_windows(n, world, rank)
    got = multigpu.pairprob_distributed(table(w0, w1) if w1 > w0 else None, W, step, rank, world, dist, n, CUTOFF)
    if rank == 0:
        ref = table(0, n).reduce(0, None, CUTOFF)
        assert len(got[0]) == len(ref[0])
        for a, b in zip(got, ref):
            assert a.dtype == b.dtype and np.array_equal(a, b)
        print("PAIRPROB_OK", len(got[1]))
    else:
        assert got is None
    dist.destroy_process_group()
""")


# 16 windows over 8 ranks: shards of 2 windows, halo rows cross several ranks; step 25 > W 20: nucleotides no window holds
@pytest.mark.parametrize("world,L,W,step", [(2, 150, 40, 1), (3, 131, 40, 7), (4, 150, 40, 1), (8, 100, 40, 4),
                                            (3, 290, 20, 25)])
def test_multi_rank_reduction_equals_one_rank(world, L, W, step, tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT, "L": L, "W": W, "step": step})
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(29100 + os.getpid() % 400), str(script)]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert p.returncode == 0, p.stdout[-3000:]
    assert "PAIRPROB_OK" in p.stdout, p.stdout[-3000:]
