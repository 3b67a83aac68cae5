"""ScanFold.py-compatible command line on the CUDA engine.

Same positional argument, flags and defaults as the reference (ScanFold.py:54-155), same output folder and
file names (ScanFold.py:310-388,1484-1500), same file contents.  Additive flags only: --seed (Philox key of
the device shuffles), --parity_shuffles (host-provided shuffles, for bit-exact comparison with a reference
run), --params (ViennaRNA .par file), --gpu (device ordinal).

The structure-extraction step that follows the ScanFold-Fold outputs (motif .dbn / .ct files and
ExtractedStructures.gff3, ScanFold.py:1557-1781) runs too, every motif as one single-window scan; only its
PostScript plots are not written.

--global_refold (three full-length folds on the blocked kernel), --by_ed, -c 0, --print and --print_random behave as in
the reference.  Not carried over (SURVEY 2, out of scope): --lri, --algo rnastructure, --fold_only, --dont_scan; selecting
one of them is an error, not a silent no-op.
"""
import argparse
import os
import random
import re
import sys
import time
from datetime import datetime

import numpy as np

from . import motifs, pipeline, scan


BESTEFFORT_WARNING = (
    "scanfold_b200: WARNING -- the built-in energy table is a BEST-EFFORT stand-in for ViennaRNA's rna_turner2004.par\n"
    "  (the real file is not redistributable from this image; stack / loop values were re-typed from the published\n"
    "  model and the 1x1, 2x1 and 2x2 interior-loop tables are rule-generated).  Energies, z-scores and structures\n"
    "  therefore differ from a ViennaRNA-backed ScanFold run.  Pass --params /path/to/rna_turner2004.par (or set\n"
    "  SCANFOLD_PARAMS) to fold with the real Turner-2004 parameters.\n")


def build_parser():
    p = argparse.ArgumentParser(prog="ScanFold.py")
    p.add_argument("filename", type=str, help="input FASTA file")
    p.add_argument("--react", type=str, help="SHAPE reactivity file (2 or 3 tab-separated columns)")
    p.add_argument("-m", type=float, default=0.8, help="SHAPE slope")
    p.add_argument("-b", type=float, default=-0.2, help="SHAPE intercept")
    p.add_argument("--shapeD", action="store_true", help="Deigan SHAPE pseudo-energies")
    p.add_argument("--shapeZ", action="store_true", help="Zarringhalam SHAPE pseudo-energies")
    p.add_argument("--name", type=str, default="UserInput", help="sequence name used as chrom in wig/bp/fa")
    p.add_argument("--fold_only", action="store_true")
    p.add_argument("--dont_scan", action="store_true")
    p.add_argument("--fold", action="store_true", default=True)
    p.add_argument("-f", type=int, default=-2, help="legacy z-score filter")
    p.add_argument("-c", type=int, default=1, help="competition on (1) or off (0)")
    p.add_argument("--out_name", type=str, default=None, help="output folder name")
    p.add_argument("-s", type=int, default=1, help="step size")
    p.add_argument("-w", type=int, default=120, help="window size")
    p.add_argument("-r", type=int, default=100, help="randomizations per window")
    p.add_argument("-t", type=int, default=37, help="temperature (C)")
    p.add_argument("--type", type=str, default="mono", help="shuffle type: mono or di")
    p.add_argument("--print", action="store_true")
    p.add_argument("--print_random", action="store_true")
    p.add_argument("--algo", type=str, default="rnafold")
    p.add_argument("--constraints", type=str, help="hard-constraint file; line 3 holds one symbol per nucleotide")
    p.add_argument("--span", type=int, help="maximum base-pair span")
    p.add_argument("--global_refold", action="store_true")
    p.add_argument("--lri", action="store_true")
    p.add_argument("--kmer", type=int, default=20)
    p.add_argument("--kmer_step_size", type=int, default=1)
    p.add_argument("--lri_cutoff", type=int, default=-25)
    p.add_argument("--by_ed", action="store_true")
    p.add_argument("--out1", type=str, default="./ScanFold.NoFilter")
    p.add_argument("--out2", type=str, default="./ScanFold.-1Filter")
    p.add_argument("--out3", type=str, default="./ScanFold.-2Filter")
    p.add_argument("--out4", type=str, default="./ScanFold.Log.txt")
    p.add_argument("--out5", type=str, default="./ScanFold.FinalPartners.txt")
    p.add_argument("--out6", type=str, default="./IGV_BP_Track")
    p.add_argument("--fasta_index", type=str, default="./user_input.fai")
    p.add_argument("--dbn_file_path", type=str, default="AllDBN-global_refold.txt")
    p.add_argument("--dbn_file_path1", type=str, default="Zavg_NoFilter")
    p.add_argument("--dbn_file_path2", type=str, default="Zavg_-1_pairs")
    p.add_argument("--dbn_file_path3", type=str, default="Zavg_-2_pairs")
    p.add_argument("--dbn_file_path4", type=str, default="AllDBN.txt")
    p.add_argument("--structure_extract_file", type=str, default="ExtractedStructures.gff3")
    p.add_argument("--final_partners_wig", type=str, default="./IGV_BP_Zavg_metrics")
    # additive
    p.add_argument("--seed", type=int, default=42, help="[scanfold_b200] Philox key for device shuffles")
    p.add_argument("--parity_shuffles", type=str, default=None,
                   help="[scanfold_b200] .npz with `shuffles` [(windows+1), r, W] uint8 to fold instead of device shuffles")
    p.add_argument("--params", type=str, default=None, help="[scanfold_b200] ViennaRNA parameter file")
    p.add_argument("--gpu", type=int, default=0, help="[scanfold_b200] CUDA device ordinal")
    p.add_argument("--pair_probs", action="store_true",
                   help="[scanfold_b200] also write the window-averaged base-pair probabilities of the scan's partition "
                        "functions: <out>.pairprob.wig (probability of being paired), <out>.pairprob.txt (pairs with "
                        "P >= 0.01) and an IGV arc track of the pairs with P >= 0.1")
    return p


def read_fasta(path):
    """records as (name, sequence); name = header up to the first whitespace (Biopython's record.name)"""
    name, chunks = None, []
    with open(path) as f:
        for line in f:
            line = line.rstrip("\n")
            if line.startswith(">"):
                if name is not None:
                    yield name, "".join(chunks)
                parts = line[1:].split()
                name, chunks = (parts[0] if parts else ""), []
            elif name is not None:
                chunks.append(line.strip())
    if name is not None:
        yield name, "".join(chunks)


def read_reactivities(path):
    """getShapeDataFromFile (ScanFold.py:218-262): 1-based list, -999 for NA and for positions the file skips"""
    vec = [-999.0]
    count = 1
    lines = open(path).read().splitlines()
    ncol = len(lines[0].split("\t"))
    if ncol not in (2, 3):
        raise ValueError("Trouble parsing reactivity data")
    for line in lines:
        f = line.split("\t")
        pos = int(f[0])
        value = f[2] if ncol == 3 else f[1]
        if value == "NA":
            value = -999
        if pos != count:
            vec.extend([-999.0] * (pos - count))
            count = pos
        vec.append(float(value))
        count += 1
    return vec


def make_output_folder(cwd, out_name, read_name):
    """folder cascade of ScanFold.py:310-369"""
    stamp = lambda: datetime.now().strftime("%m-%d-%Y-%H.%M.%S")
    rnd3 = lambda: str(random.randint(100, 999))
    try:
        if out_name is not None:
            try:
                folder = out_name
                os.mkdir(os.path.join(cwd, folder))
            except OSError:
                folder = out_name + "_" + stamp()
                os.mkdir(os.path.join(cwd, folder))
        else:
            folder = read_name
            os.mkdir(os.path.join(cwd, folder))
    except OSError:
        try:
            folder = (out_name + "_" + stamp() + "_" + rnd3()) if out_name is not None else "SF_Results_" + stamp()
            os.mkdir(os.path.join(cwd, folder))
        except OSError:
            folder = "ScanFold-Results_" + stamp() + "_" + rnd3()
            os.mkdir(os.path.join(cwd, folder))
    print("Making output folder named:" + folder)
    return folder


def emit_window_prints(args, seq, table, react, hc, temperature):
    """What the reference prints per window, in window order: the reactivity slice in the SHAPE branch
    (ScanFold.py:524), the energy list under --print_random (:551-552) and the result row under --print (:680-684)."""
    if react is None and not args.print_random and not args.print:
        return
    from . import engine, stats, writers
    W, step = table.W, table.step
    db = engine.pair_tables_to_dotbrackets(table.pair_tbl) if args.print else None
    cen = engine.pair_tables_to_dotbrackets(table.centroid_tbl) if args.print else None
    for k in range(len(table)):
        s1, e1 = int(table.start1[k]), int(table.end1[k])
        if react is not None:
            print(react[s1:e1 + 1])
        if args.print_random:
            row = np.concatenate([[table.native_unconstrained_dcal[k]], table.shuffle_dcal[k]])
            print([float(x) for x in stats.energy_to_float(row)])
        if args.print:
            frag = seq[s1 - 1:e1]
            cols = [s1, e1, temperature, float(table.mfe[k]), float(table.z[k]), float(table.p[k]), float(table.ed[k])]
            if hc is not None:
                print("\t".join(str(c) for c in cols) + "\n" + frag + "\n" + hc[s1 - 1:e1] + "\n" + db[k] + "\n" + cen[k] +
                      str(writers.gc_content(frag)) + "\n")
            else:
                print("\t".join(str(c) for c in cols + [frag, db[k], cen[k], writers.gc_content(frag)]) + "\n")


def global_refold(seq, names, name, temperature, max_span):
    """--global_refold (ScanFold.py:1509-1551): the whole record folded three times -- with the Zavg < -1 pairs as hard
    constraints, with the Zavg < -2 pairs, and unconstrained -- and written to the refold dbn file.  Line 3 of a Zavg dbn
    file covers the nucleotides the scan covered; ViennaRNA applies a shorter constraint string to the leading positions."""
    from . import engine
    print("Refolding full sequence using ScanFold results as constraints...")
    out = []
    for path in (names.dbn2, names.dbn3):
        hc = open(path + ".dbn").readlines()[2].rstrip("\n")
        out.append(engine.fold_long(seq.upper(), hc=hc, temperature=temperature, max_span=max_span))
    full = engine.fold_long(seq.upper(), temperature=temperature, max_span=max_span)
    f32 = lambda e: str(float(np.float32(e / 100.0)))          # vrna_mfe returns a C float
    db = lambda pt: engine.pair_table_to_dotbracket(pt)
    with open(names.dbn_refold, "w") as f:
        f.write(">%s\tGlobal Full MFE=%s\n%s\n%s\n" % (name, f32(full[0]), seq, db(full[1])))
        f.write(">%s\tRefolded with -1 constraints MFE=%s\n%s\n%s\n" % (name, f32(out[0][0]), seq, db(out[0][1])))
        f.write(">%s\tRefolded with -2 constraints MFE=%s\n%s\n%s\n" % (name, f32(out[1][0]), seq, db(out[1][1])))


def run_record(args, record_name, raw_seq, original_directory, dist=None):
    """One FASTA record.  With a torch.distributed process group (torchrun, one process per GPU) the windows are
    sharded by range over the ranks; rank 0 owns the output folder and writes every file."""
    from . import engine, multigpu
    t0 = time.time()
    rank = dist.get_rank() if dist is not None else 0
    world = dist.get_world_size() if dist is not None else 1
    seq = raw_seq.replace("T", "U").replace("t", "u")      # Seq.transcribe (ScanFold.py:282)
    if "-" in seq:
        raise ValueError("Gaps found in sequence. Please submit a complete sequence to ScanFold")
    read_name = record_name
    if "|" in read_name:
        read_name = re.split(r"\|", read_name)[0]
    cwd = os.getcwd()
    folder = None
    if rank == 0:
        folder = make_output_folder(cwd, args.out_name, read_name)
        os.chdir(os.path.join(cwd, folder))
    try:
        W, step, r = int(args.w), int(args.s), int(args.r)
        names = pipeline.RunNames(read_name, record_name, W, step, r, str(args.type), name=args.name, out6=args.out6,
                                  final_partners_wig=args.final_partners_wig, dbn1=args.dbn_file_path1,
                                  dbn2=args.dbn_file_path2, dbn3=args.dbn_file_path3, dbn4=args.dbn_file_path4,
                                  out1=args.out1, out2=args.out2, out3=args.out3, dbn_refold=args.dbn_file_path)
        if rank == 0:
            print("Output name=" + names.outname)
        if len(seq) < W:
            if rank == 0:
                print(record_name + " sequence is less than window size. Moving on to next entry.")
            return
        hc = None
        if args.constraints is not None:
            # opened after the chdir into the output folder in the reference (Appendix B Q8): a relative path is looked
            # up in the freshly made folder and fails there; every rank takes the same decision before any collective
            if not os.path.isabs(args.constraints):
                raise FileNotFoundError("[Errno 2] No such file or directory: %r (the reference opens --constraints "
                                        "from inside the output folder: give an absolute path)" % args.constraints)
            if rank == 0:
                print("Considering constraint input")
            hc = open(args.constraints).readlines()[2].rstrip("\n")
        react = None
        if args.react is not None:
            if rank == 0:
                print("Considering SHAPE reactivity input")
            react = read_reactivities(os.path.join(original_directory, args.react))
            if hc is not None:
                react = None       # ScanFold.py:508-519: the constraints branch wins, the reactivities are never applied
            elif args.shapeZ and not args.shapeD:
                raise TypeError("sc_add_SHAPE_zarringhalam() is called with one argument by the reference "
                                "(ScanFold.py:536) and fails there too; use --shapeD")
        total = scan.n_windows_of(len(seq), W, step)
        w0, w1 = multigpu.shard_windows(total, world, rank)
        last = w1 == total and w1 > w0
        parity = None
        if args.parity_shuffles:
            allsh = np.load(args.parity_shuffles if os.path.isabs(args.parity_shuffles)
                            else os.path.join(original_directory, args.parity_shuffles))["shuffles"]
            parity = allsh[w0:w1 + (1 if last else 0)]
        if rank == 0:
            print("Scanning input sequence:", read_name)
        acc = pp = None
        if w1 > w0:
            if args.pair_probs:
                pp = engine.PairProbTable(len(seq), W, step, w0, w1 - w0)
            shard = scan.scan_record(seq.upper(), W, step, r, shuffle_type=str(args.type), seed=args.seed,
                                     parity_shuffles=parity, temperature=float(args.t), max_span=args.span or 0, hc=hc,
                                     react=react, shape_m=args.m, shape_b=args.b, first_window=w0, n_windows=w1 - w0,
                                     final_window=last, pairprob=pp)
            shard.alln = scan.all_n_windows(seq, W, step, w0, w1 - w0)      # Q10: tested on the record as given
            if last and scan.final_window_all_n(seq, W):
                shard.final = None                                          # the final-window block appends nothing (:719-726)
            z100, mfe100, ed100 = pipeline.fold_inputs(shard)
            acc = engine.Accumulator(len(seq), W, step, w0, shard.pair_tbl, z100, mfe100, ed100, skip=shard.alln)
        else:                  # more ranks than windows: this rank only takes part in the collectives
            shard = scan.empty_table(W, step, r, w0)
        try:
            own_table = multigpu.own_partner_table(acc, W, step, rank, world, dist, total)
        finally:
            if acc is not None:
                acc.close()
        pairprob = None
        if args.pair_probs:
            try:
                pairprob = multigpu.pairprob_distributed(pp, W, step, rank, world, dist, total, engine.PAIR_CUTOFF)
            finally:
                if pp is not None:
                    pp.close()
        # every rank aggregates the nucleotides it owns; rank 0 gets the per-nucleotide results and the log text
        aggregated = multigpu.aggregate_distributed(own_table, seq, rank, world, dist, by_ed=bool(args.by_ed), with_logs=True)
        table = multigpu.gather_window_tables(shard, rank, world, dist, with_shuffle_energies=bool(args.print_random))
        if rank != 0:
            return
        emit_window_prints(args, seq, table, react, hc, int(args.t))
        minz = pipeline.write_scan_outputs(seq, table, names, int(args.t), step)   # Sequence column keeps input case (Q11)
        print("Elapsed time: %ss" % round(time.time() - t0, 2))
        print("Determining best base pairs...")
        pipeline.write_fold_outputs(seq, None, names, minz, step, by_ed=bool(args.by_ed), competition=int(args.c),
                                    zscores=pipeline.zscore_total(table), filter_value=int(args.f),
                                    input_filename=args.filename, aggregated=aggregated)
        if pairprob is not None:
            pipeline.write_pairprob_outputs(pairprob, names, W, step, total)
        if args.global_refold:
            global_refold(seq, names, args.name, float(args.t), args.span or 0)
        # structure extraction: refold every top-level helix of the Zavg < -2 structure (ScanFold.py:1557-1781)
        parity_npz = None
        if args.parity_shuffles:
            parity_npz = np.load(args.parity_shuffles if os.path.isabs(args.parity_shuffles)
                                 else os.path.join(original_directory, args.parity_shuffles))
        motifs.run(seq, names.dbn3 + ".dbn", args.name, args.structure_extract_file, shuffle_type=str(args.type),
                   temperature=float(args.t), seed=args.seed, parity=parity_npz)
        print("Total runtime: %ss" % round(time.time() - t0, 2))
        print("ScanFold-Fold analysis complete! Output found in folder named: " + folder)
    finally:
        os.chdir(original_directory)


def main(argv=None):
    args = build_parser().parse_args(argv)
    for flag, why in ((args.lri, "--lri (experimental duplex scan)"),
                      (str(args.algo) != "rnafold", "--algo " + str(args.algo)),
                      (args.fold_only, "--fold_only"), (args.dont_scan, "--dont_scan")):
        if flag:
            raise SystemExit("scanfold_b200: %s is outside the scanning hot path this build covers (see DESIGN.md)" % why)
    if str(args.type) not in ("mono", "di"):
        raise SystemExit('Shuffle type not properly designated; please input "di" or "mono"')
    from . import engine
    dist = None
    device = args.gpu
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:       # torchrun: one process per GPU, windows sharded by range
        import torch
        import torch.distributed as dist
        device = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(device)
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))
    engine.init(device, args.params)
    if dist is not None:       # NCCL orders its work against torch's current stream: run the library on that stream too
        engine.set_stream(torch.cuda.current_stream().cuda_stream)
    if engine.params_besteffort() and (dist is None or dist.get_rank() == 0):
        sys.stderr.write(BESTEFFORT_WARNING)
    original_directory = os.getcwd()
    if dist is None or dist.get_rank() == 0:
        print(original_directory)
    for record_name, raw_seq in read_fasta(args.filename):
        run_record(args, record_name, raw_seq, original_directory, dist)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
