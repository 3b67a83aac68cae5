"""One FASTA record through scan -> ScanFold-Fold -> output files: the body of the record loop
ScanFold.py:266-1554 (without the opt-in global refold / LRI branches), batched.

  scan        scan.scan_record            (CUDA: folds, shuffles, partition function)
  accumulate  engine.Accumulator          (CUDA: per-nucleotide partner sums)
  fold step   foldstep.aggregate/compete  (host: argmin, competition)
  outputs     writers.*                   (host: byte-identical text files)
"""
import os

import numpy as np

from . import foldstep, writers


def fold_inputs(table):
    """per-window integers the accumulator takes: round(z*100), MFE in dcal (== round(MFE, 2) * 100), round(ED*100)"""
    z100 = np.rint(np.asarray(table.z) * 100.0).astype(np.int32)
    ed100 = np.rint(np.asarray(table.ed) * 100.0).astype(np.int32)
    return z100, np.asarray(table.mfe_dcal, dtype=np.int32), ed100


def partner_table_gpu(L, table):
    """ScanFold.py:564-677 + :1051-1139 on the device -> foldstep.PartnerTable"""
    from . import engine
    z100, mfe100, ed100 = fold_inputs(table)
    acc = engine.Accumulator(L, table.W, table.step, table.first_window, table.pair_tbl, z100, mfe100, ed100,
                             skip=getattr(table, "alln", None))
    try:
        return foldstep.table_from_compact(*acc.compact(), nt0=acc.nt0)
    finally:
        acc.close()


class RunNames:
    """file names of a record's outputs (ScanFold.py:370-388,1484-1500)"""

    def __init__(self, read_name, record_name, W, step, r, shuffle_type, name="UserInput", out6="./IGV_BP_Track",
                 final_partners_wig="./IGV_BP_Zavg_metrics", dbn1="Zavg_NoFilter", dbn2="Zavg_-1_pairs",
                 dbn3="Zavg_-2_pairs", dbn4="AllDBN.txt", out1="./ScanFold.NoFilter", out2="./ScanFold.-1Filter",
                 out3="./ScanFold.-2Filter", dbn_refold="AllDBN-global_refold.txt"):
        self.out1, self.out2, self.out3, self.dbn_refold = out1, out2, out3, dbn_refold
        self.read_name, self.record_name, self.name = read_name, record_name, name
        self.outname = "%s.win_%d.stp_%d.rnd_%d.shfl_%s" % (read_name, W, step, r, shuffle_type)
        self.out6, self.final_partners_wig = out6, final_partners_wig
        self.dbn1, self.dbn2, self.dbn3, self.dbn4 = dbn1, dbn2, dbn3, dbn4


def write_pairprob_outputs(pairprob, names, W, step, total_windows):
    """the three files of --pair_probs: paired(i) track, pair list (P >= 0.01), IGV arcs (P >= 0.1)"""
    from . import engine
    paired, i, j, p = pairprob
    pos = np.arange(len(paired))
    covered = engine.windows_holding(pos, pos, W, step, total_windows) > 0
    o = names.outname
    writers.write_pairprob_wig(o + ".pairprob.wig", paired, covered, names.name)
    writers.write_pairprob_txt(o + ".pairprob.txt", i, j, p)
    writers.write_pairprob_bp(names.out6 + "." + o + ".pairprob.bp", i, j, p, names.name)


def zscore_total(table):
    """the reference's zscore_total (ScanFold.py:556,751): every numeric z of the scan loop plus the final-window one"""
    alln = table.alln if getattr(table, "alln", None) is not None else np.zeros(len(table), dtype=bool)
    z = table.z[~alln].tolist()
    return z + ([table.final["z"]] if table.final is not None else [])


def write_scan_outputs(seq, table, names, temperature, step):
    """.out table and the four scan wig tracks (ScanFold.py:416,685,1495-1499); returns minz (:766)"""
    o = names.outname
    writers.write_out(o + ".out", names.read_name, seq, table, temperature)
    fin = table.final
    alln = table.alln if getattr(table, "alln", None) is not None else np.zeros(len(table), dtype=bool)
    extra = (lambda key: [fin[key]]) if fin is not None else (lambda key: [])

    def track(values, all_n_value):
        lst = values.tolist()
        for k in np.nonzero(alln)[0]:                 # Q10: int 0 / "#DIV/0" entries of the all-N short-circuit
            lst[k] = all_n_value
        return lst

    writers.write_wig(o + ".scan-MFE.wig", track(table.mfe, 0) + extra("mfe"), step, names.name)
    writers.write_wig(o + ".scan-zscores.wig", track(table.z, "#DIV/0") + extra("z"), step, names.name)
    writers.write_wig(o + ".scan-pvalue.wig", track(table.p, 0) + extra("p"), step, names.name)
    writers.write_wig(o + ".scan-ED.wig", track(table.ed, 0) + extra("ed"), step, names.name)
    zt = zscore_total(table)
    if not zt:
        raise ValueError("no window produced a z-score (every window is all-N): statistics.mean of an empty list "
                         "fails in the reference too (ScanFold.py:761)")
    return min(zt)


def write_fold_outputs(seq, ptable, names, minz, step, by_ed=False, competition=1, zscores=None, filter_value=-2,
                       input_filename="", aggregated=None):
    """ScanFold-Fold: logs, CT / dbn / bp / wig / fasta files (ScanFold.py:1036-1500,1554).  Returns (agg, final).
    by_ed: --by_ed (ED-weighted partner choice and log names, :380-385,1190-1215).  competition = 0: the -c 0 branch
    (:1454-1466): .dp files instead of CT / dbn / bp, then the reference dies opening the missing dbn file -- so do we.
    aggregated: (NtResult, log text, pair-count text) when the ranks of a multi-GPU run aggregated their own nucleotides
    (multigpu.aggregate_distributed); ptable is not needed then."""
    import statistics
    o = names.outname
    tag = ".ScanFold.ED-weighted" if by_ed else ".ScanFold"
    with open(o + tag + ".log", "w") as log_total, open(o + ".ntPairCounts.log", "w") as sirna:
        sirna.write("i\tnuc\twindows\tbps\n")
        if aggregated is not None:
            agg = aggregated[0]
            log_total.write(aggregated[1])
            sirna.write(aggregated[2])
        else:
            agg = foldstep.aggregate(ptable, seq, log_total, sirna, by_ed=by_ed)
    key = agg.coord
    if competition == 0:
        with open(o + tag + ".FinalPartners.txt", "w") as log_win:
            log_win.write(foldstep.FINAL_PARTNERS_HEADER)
        meanz = float(statistics.mean(zscores))
        one_sig_below = float(meanz - float(statistics.stdev(zscores)))
        print("Writing DP files, can not write CT files...")
        writers.write_bp(names.out6 + "." + o + names.record_name + ".ALL.bp", key, agg.part, agg.mean_z, names.name, minz,
                         coord=key)
        output = names.read_name + "." + str(input_filename) + ".ScanFold."
        dp = lambda path, filt: writers.write_dp(path, key, key, agg.part, agg.mean_z, filt, minz)
        if filter_value is not None:
            dp(output + str(filter_value) + names.record_name + ".dp", filter_value)
        dp(names.out1 + "." + o + ".dp", float(10))
        dp(names.out2 + "." + o + ".dp", float(-1))
        dp(names.out3 + "." + o + ".dp", float(-2))
        dp(output + "." + o + "mean_" + str(round(meanz, 2)) + ".dp", meanz)
        dp(output + "." + o + "below_mean_" + str(round(one_sig_below, 2)) + ".dp", one_sig_below)
        print("ScanFold-Fold complete, find results in...")
        writers.write_fasta(names.name + "." + o + ".fa", seq, names.name)
        open(names.dbn4, "w").close()     # `cat` of three dbn files that were never written (ScanFold.py:1554)
        return agg, None
    with open(o + tag + ".FinalPartners.txt", "w") as log_win:
        fin = foldstep.compete(agg, seq, log_win)
    covered = "".join(seq[k - 1] for k in key.tolist())
    dbn_text = []
    for path, filt, title in ((names.dbn1, 10.0, "NoFilter"), (names.dbn2, -1.0, "Zavg_-1"), (names.dbn3, -2.0, "Zavg_-2")):
        partner = writers.write_ct(path + ".ct", fin, seq, filt, names.name)
        writers.write_dbn(path + ".dbn", title, covered, partner, key)
        dbn_text.append(open(path + ".dbn").read())
    writers.write_bp(names.out6 + "." + o + ".bp", fin.i, fin.j, fin.z, names.name, minz, coord=key)
    writers.write_wig_dict(names.final_partners_wig + "." + o + ".wig", fin.z, names.name, step)
    writers.write_bp(names.out6 + "." + o + "." + names.record_name + ".ALL.bp", key, agg.part, agg.mean_z, names.name,
                     minz, coord=key)
    writers.write_fasta(names.name + "." + o + ".fa", seq, names.name)
    with open(names.dbn4, "w") as f:      # `cat` of the three dbn files (ScanFold.py:1554)
        f.write("".join(dbn_text))
    return agg, fin
