"""Output files of a ScanFold run, byte-identical to the reference writers:
  .out rows            ScanFold.py:416,685          write_ct       ScanFoldFunctions.py:476-518
  makedbn              ScanFoldFunctions.py:67-138  write_bp       :644-712
  write_wig            :626-642                     write_wig_dict :616-624
  write_fasta          :597-605
and the additive pair-probability files of --pair_probs (write_pairprob_*), which have no reference counterpart.
The reference's CT files can be asymmetric (i -> j while j -> 0, Appendix B Q14); makedbn's '<' / '>'
symbols for non-nested partners are reproduced from the CT rows, not from a pair table.
"""
import numpy as np


def gc_content(frag):
    """get_gc_content (ScanFoldFunctions.py:1023-1035) including its `'C' and 'G' in frag` quirk (Q9)"""
    if "G" in frag:
        a = frag.count("A") + frag.count("a")
        g = frag.count("G") + frag.count("g")
        c = frag.count("C") + frag.count("c")
        t = frag.count("T") + frag.count("t") + frag.count("U") + frag.count("u")
        return round(float(g + c) / float(a + t + g + c), 5)
    return 0


ALL_N_STRUCTURE = "." * 120      # the literal 120-dot strings of ScanFold.py:490-491


def write_out(path, read_name, seq, table, temperature):
    """the per-window table: header ScanFold.py:416, rows :685.  Windows the reference short-circuits as all-N
    (Appendix B Q10: a literal 120-character comparison, :486-492) print MFE 0, z "#DIV/0", p 0, ED 0 and 120 dots."""
    W = table.W
    rows = ["i\tj\tTemperature\tNative_dG\tZ-score\tP-score\tEnsembleDiversity\tSequence\tStructure\tCentroid\t"
            + read_name + "\n"]
    from .engine import pair_tables_to_dotbrackets
    n = len(table)
    structures = pair_tables_to_dotbrackets(table.pair_tbl[:n])
    centroids = pair_tables_to_dotbrackets(table.centroid_tbl[:n])
    alln = table.alln if getattr(table, "alln", None) is not None else np.zeros(n, dtype=bool)
    for k in range(n):
        s0 = int(table.start1[k]) - 1
        frag = seq[s0:s0 + W]
        if alln[k]:
            rows.append("%d\t%d\t%s\t0\t#DIV/0\t0\t0\t%s\t%s\t%s\t%s\n" % (
                table.start1[k], table.end1[k], str(temperature), frag, ALL_N_STRUCTURE, ALL_N_STRUCTURE,
                str(gc_content(frag))))
            continue
        rows.append("%d\t%d\t%s\t%s\t%s\t%s\t%s\t%s\t%s\t%s\t%s\n" % (
            table.start1[k], table.end1[k], str(temperature), str(float(table.mfe[k])), str(float(table.z[k])),
            str(float(table.p[k])), str(float(table.ed[k])), frag, structures[k], centroids[k],
            str(gc_content(frag))))
    with open(path, "w") as f:
        f.write("".join(rows))


def write_wig(path, values, step, name):
    """write_wig (ScanFoldFunctions.py:626-641): "%f" per value; a string entry (the "#DIV/0" z-score of an all-N window)
    falls through to "%s" """
    with open(path, "w") as f:
        f.write("fixedStep chrom=%s start=1 step=%s span=%s\n" % (name, step, step))
        f.write("".join(("%s\n" % v) if isinstance(v, str) else ("%f\n" % v) for v in values))


def ct_rows(fin, seq, filt):
    """partner column of write_ct(final_partners, ..., filter, strand=1, ...) for every covered nucleotide"""
    n = len(fin.i)
    key = fin.coord
    passed = fin.z < filt
    partner = np.zeros(n, dtype=np.int64)
    is_i = fin.i == key
    is_j = (fin.j == key) & ~is_i
    paired = fin.i != fin.j
    partner[passed & paired & is_i] = fin.j[passed & paired & is_i]
    partner[passed & paired & is_j] = fin.i[passed & paired & is_j]
    bad = ~(is_i | is_j)
    if bad.any():
        raise ValueError("WriteCT function did not find a nucleotide to match coordinate")
    # nucleotide column: v.inucleotide when key == i, v.jnucleotide when key == j
    return partner


def write_ct(path, fin, seq, filt, name):
    partner = ct_rows(fin, seq, filt)
    n = len(partner)
    rows = ["%d\t%s\n" % (n, name)]
    rows.extend("%d %s %d %d %d %d\n" % (k, seq[k - 1], k - 1, k + 1, partner[r], k) for r, k in enumerate(fin.coord.tolist()))
    with open(path, "w") as f:
        f.write("".join(rows))
    return partner


def dbn_string(partner, coord=None):
    """makedbn's symbol per CT row (ScanFoldFunctions.py:67-130): partner[r] = CT column 5 of row r, coord[r] its
    coordinate.  The reference looks the partner up by slicing the file at LINE number icoord, which is the row of
    coordinate icoord only while no nucleotide is missing from the table; the slice is reproduced as is."""
    n = len(partner)
    p = partner.tolist()
    c = list(range(1, n + 1)) if coord is None else list(coord)
    out = []
    for r in range(n):
        i, j = c[r], p[r]
        if j == 0:
            out.append(".")
        elif i < j:
            sym = None
            for q in range(i - 1, n):           # data[icoord:] with data[0] = the header line
                if c[q] == j:
                    sym = "("
                    break
                if p[q] != 0 and p[q] < i:
                    sym = "<"
                    break
            if sym:
                out.append(sym)
        elif i > j:
            sym = None
            for q in range(j - 1, n):
                if c[q] == i:
                    sym = ")"
                    break
                if p[q] != 0 and p[q] < j:
                    sym = ">"
                    break
            if sym:
                out.append(sym)
    return "".join(out)


def write_dbn(path, title, seq_covered, partner, coord=None):
    with open(path, "w") as f:
        f.write(">%s\n%s\n%s\n" % (title, seq_covered, dbn_string(partner, coord)))


def _bp_score(z):
    if z < -2.0:
        return "0"
    if z < -1 and z >= -2:
        return "1"
    if z < 0 and z >= -1:
        return "2"
    if z == 0:
        return "3"
    if 0 < z <= 1:
        return "4"
    if 1 < z <= 2:
        return "5"
    if z > 2:
        return "6"
    raise ValueError("write_bp: z-score %r has no colour class" % (z,))


def write_dp(path, coord, i_arr, j_arr, z_arr, filt, minz):
    """write_dp (ScanFoldFunctions.py:564-578), the IGV .dp files of a -c 0 run: one line per entry with z < filter"""
    rows = []
    for k, i, j, z in zip(coord.tolist(), i_arr.tolist(), j_arr.tolist(), z_arr.tolist()):
        if float(z) < filt:
            rows.append("%d\t%d\t%f\n" % (k if i == j else i, j, float((-1 / minz) * z) / minz))
    with open(path, "w") as f:
        f.write("".join(rows))


def write_bp(path, i_arr, j_arr, z_arr, name, minz, coord=None):
    rows = ["color:\t55\t129\t255\tLess than -2 %s\n" % str(minz), "color:\t89\t222\t111\t-1 to -2\n",
            "color:\t236\t236\t136\t0 to -1\n", "color:\t199\t199\t199\t0\n", "color:\t228\t228\t228\t0 to 1\n",
            "color:\t243\t243\t243\t1 to 2\n", "color:\t247\t247\t247\tGreater than 2\n"]
    il, jl, zl = i_arr.tolist(), j_arr.tolist(), z_arr.tolist()
    for k0 in range(len(il)):
        i, j = il[k0], jl[k0]
        if i == j:
            i = k0 + 1 if coord is None else int(coord[k0])   # the unpaired branch prints the dictionary key
        rows.append("%s\t%d\t%d\t%d\t%d\t%s\n" % (name, i, i, j, j, _bp_score(zl[k0])))
    with open(path, "w") as f:
        f.write("".join(rows))


def write_wig_dict(path, z_arr, name, step):
    with open(path, "w") as f:
        f.write("fixedStep chrom=%s start=1 step=%s span=%s\n" % (name, step, step))
        f.write("".join("%f\n" % v for v in z_arr.tolist()))


def write_pairprob_wig(path, paired, covered, name):
    """paired(i) per nucleotide as a variableStep track; nucleotides no window holds (covered False) are left out"""
    pos = np.nonzero(covered)[0]
    with open(path, "w") as f:
        f.write("variableStep chrom=%s span=1\n" % name)
        f.write("".join("%d\t%f\n" % (k + 1, v) for k, v in zip(pos.tolist(), np.asarray(paired)[pos].tolist())))


def write_pairprob_txt(path, i_arr, j_arr, p_arr):
    """the listed pairs, 1-based, sorted by i then j"""
    with open(path, "w") as f:
        f.write("i\tj\tprobability\n")
        f.write("".join("%d\t%d\t%.6f\n" % r for r in zip(i_arr.tolist(), j_arr.tolist(), p_arr.tolist())))


PAIRPROB_BP_CLASSES = ((0.1, "color:\t199\t199\t199\t0.1 to 0.3\n"), (0.3, "color:\t236\t236\t136\t0.3 to 0.5\n"),
                       (0.5, "color:\t89\t222\t111\t0.5 to 0.8\n"), (0.8, "color:\t55\t129\t255\t0.8 to 1\n"))


def write_pairprob_bp(path, i_arr, j_arr, p_arr, name):
    """IGV arc track in the layout of write_bp: the pairs with P >= 0.1, colour class = the last column"""
    lows = np.array([c[0] for c in PAIRPROB_BP_CLASSES])
    p_arr = np.asarray(p_arr)
    keep = p_arr >= lows[0]
    cls = np.searchsorted(lows, p_arr[keep], side="right") - 1
    rows = [c[1] for c in PAIRPROB_BP_CLASSES]
    rows += ["%s\t%d\t%d\t%d\t%d\t%d\n" % (name, i, i, j, j, c)
             for i, j, c in zip(np.asarray(i_arr)[keep].tolist(), np.asarray(j_arr)[keep].tolist(), cls.tolist())]
    with open(path, "w") as f:
        f.write("".join(rows))


def write_fasta(path, seq, name):
    with open(path, "w") as f:
        f.write(">%s\n%s\n" % (name, seq))
