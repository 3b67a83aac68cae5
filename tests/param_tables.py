"""Seeded energy-table families for parity tests at the edges of the table space.

Every family rewrites the shipped stand-in parameter file (ViennaRNA v2.0 format) into a new file.  The kernels take
shortcuts that depend on table shape -- int16 storage, packed 10-bit mismatch fields, the stencil / range-minimum split
of the asymmetry penalty, special-loop lookups -- so the tests fold under tables that push each of those.

    uniform(seed)        every numeric entry random in [-300, 300] (INF stays INF), NINIO m in [0, 120], max in [0, 5m]
    coarse(seed)         like uniform, every value a multiple of 100: co-optimal structures, traceback order matters
    favour(cls)          stand-in tables with one loop class made dominant (FAVOUR_CLASSES)
    inf(seed)            ~5 % of the stack / mismatch / dangle / int11 / int21 / int22 entries become INF
    stack_scaled(k)      stand-in with `stack` multiplied by k: folds below the int16 kernels' -12000 dcal bound
    declined(variant)    'ninio': 5 * ninio < max_ninio (mfe3 / mfe2 decline); 'mismatch': a mismatch_interior entry
                         of 600, beyond the blocked kernel's 10-bit field (mfe4 declines)
"""
import os
import random

STANDIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scanfold_b200", "params",
                       "rna_turner2004_besteffort.par")
SPECIAL = ("Tetraloops", "Triloops", "Hexaloops")
FAVOUR_CLASSES = ("hairpin", "bulge", "interior", "ninio", "mlbase", "mlintern", "terminal_au", "special")
INF_BLOCKS = ("stack", "mismatch_hairpin", "mismatch_interior", "mismatch_interior_1n", "mismatch_interior_23",
              "mismatch_multi", "mismatch_exterior", "dangle5", "dangle3", "int11", "int21", "int22")
# mfe4.cu packs interior mismatches into 10-bit fields with a bias of FB = 512 (mfe4.cu, mfe4_upload_tables: fits10)
MFE4_FIELD = 512


def _is_num(t):
    return t == "INF" or t.lstrip("-").replace(".", "", 1).isdigit()


class Table:
    """The parameter file as blocks of numbers: blocks[name] = list of rows (ints, None for INF; floats kept)."""

    def __init__(self, path=STANDIN):
        self.lines = open(path).read().split("\n")
        self.blocks = {}
        self._where = []            # (line index, block, row index) of every numeric / special row
        name = None
        for k, line in enumerate(self.lines):
            if line.startswith("# "):
                name = line[2:].strip()
                self.blocks[name] = []
                continue
            toks = line.split()
            if not toks or name is None or line.lstrip().startswith(("/*", "#")):
                continue
            if name in SPECIAL:
                row = [toks[0]] + [int(t) for t in toks[1:]]
            elif all(_is_num(t) for t in toks):
                row = [None if t == "INF" else (float(t) if "." in t else int(t)) for t in toks]
            else:
                continue
            self._where.append((k, name, len(self.blocks[name])))
            self.blocks[name].append(row)

    def write(self, path):
        out = list(self.lines)
        for k, name, r in self._where:
            row = self.blocks[name][r]
            out[k] = " ".join("INF" if v is None else (("%.6f" % v) if isinstance(v, float) else str(v)) for v in row)
        with open(path, "w") as f:
            f.write("\n".join(out))
        return str(path)

    def entries(self, names):
        """(block, row, col) of every finite integer entry of the named blocks"""
        for name in names:
            for r, row in enumerate(self.blocks.get(name, [])):
                for c, v in enumerate(row):
                    if isinstance(v, int) and not isinstance(v, bool):
                        yield name, r, c

    def get(self, name, r, c):
        return self.blocks[name][r][c]

    def set(self, name, r, c, v):
        self.blocks[name][r][c] = v

    def set_flat(self, name, idx, v):
        """entry `idx` of a block in file order (the loop-size blocks hold sizes 0..30 in rows of ten)"""
        for row in self.blocks[name]:
            if idx < len(row):
                row[idx] = v
                return
            idx -= len(row)
        raise IndexError(name)

    # scalar blocks (one row each)
    def ml(self):
        return dict(zip(("MLbase", "MLbase_dH", "MLclosing", "MLclosing_dH", "MLintern", "MLintern_dH"), self.blocks["ML_params"][0]))

    def ninio(self):
        m, _, mx = self.blocks["NINIO"][0]
        return m, mx

    def special_keys(self):
        return [row[0] for name in SPECIAL for row in self.blocks.get(name, [])]


def _randomise(t, rng, draw):
    numeric = [n for n in t.blocks if n not in SPECIAL and n not in ("NINIO", "Misc")]
    for name, r, c in t.entries(numeric):
        t.set(name, r, c, draw())
    m = draw(lo=0, hi=120)
    t.blocks["NINIO"][0] = [m, draw(), draw(lo=0, hi=5 * m)]
    misc = t.blocks["Misc"][0]
    t.blocks["Misc"][0] = [draw(), draw(), draw(), draw(), float(rng.randrange(50, 151))] + misc[5:]
    for name in SPECIAL:
        for row in t.blocks.get(name, []):
            row[1:] = [draw() for _ in row[1:]]
    return t


def uniform(seed):
    rng = random.Random(seed)
    return _randomise(Table(), rng, lambda lo=-300, hi=300: rng.randint(lo, hi))


def coarse(seed):
    rng = random.Random(seed)
    return _randomise(Table(), rng, lambda lo=-300, hi=300: 100 * rng.randint(-(-lo // 100), hi // 100))


def favour(cls):
    t = Table()
    if cls == "hairpin":
        t.set_flat("hairpin", 30, -600)                     # long hairpins through the lxc extrapolation
    elif cls in ("bulge", "interior"):
        name = "bulge" if cls == "bulge" else "interior"
        for u in (1, 2, 5, 6, 7, 30):
            t.set_flat(name, u, -500)
    elif cls == "ninio":
        t.blocks["NINIO"][0][0] = 0
        t.blocks["NINIO"][0][2] = 0
    elif cls == "mlbase":
        t.blocks["ML_params"][0][0] = -100
    elif cls == "mlintern":
        t.blocks["ML_params"][0][4] = -300
    elif cls == "terminal_au":
        t.blocks["Misc"][0][2] = -200
    elif cls == "special":
        for name in SPECIAL:
            for row in t.blocks[name]:
                row[1] = -1500
    else:
        raise ValueError(cls)
    return t


def inf(seed, frac=0.05):
    rng = random.Random(seed)
    t = Table()
    for name, r, c in t.entries(INF_BLOCKS):
        if rng.random() < frac:
            t.set(name, r, c, None)
    return t


def stack_scaled(k):
    t = Table()
    for name, r, c in t.entries(["stack"]):
        t.set(name, r, c, t.get(name, r, c) * k)
    return t


def declined(variant):
    t = Table()
    if variant == "ninio":
        t.blocks["NINIO"][0][0] = 20                       # 5 * 20 < 300 = max_ninio
    elif variant == "mismatch":
        t.set("mismatch_interior", 1, 1, 600)
    else:
        raise ValueError(variant)
    return t


# ---- the conditions the fast kernels put on a table, mirrored from their upload functions
def flat(t, name):
    """the values of a block in file order, as the loaders read them (INF -> None)"""
    return [v for row in t.blocks[name] for v in row]


def _int16_entries(t):
    """the values mfe3.cu / mfe2.cu store as int16 (their *_upload_tables, 37 C): stack, TerminalAU, the hairpin /
    interior mismatches, the multiloop-closing and stem terms, the exterior stem terms, bulge[1], interior[5] + ninio,
    MLbase and the asymmetry penalties of 1..4 nucleotides.  Mismatch / dangle blocks hold pair types 1..7."""
    ml = t.ml()
    tau, m, mx = t.blocks["Misc"][0][2], t.ninio()[0], t.ninio()[1]
    out = list(flat(t, "stack")[:49]) + [tau]
    for name in ("mismatch_hairpin", "mismatch_interior", "mismatch_interior_1n", "mismatch_interior_23"):
        out += flat(t, name)[:175]
    mm_m, mm_e = flat(t, "mismatch_multi")[:175], flat(t, "mismatch_exterior")[:175]
    d5, d3 = flat(t, "dangle5")[:35], flat(t, "dangle3")[:35]
    clip = lambda v: None if v is None else min(0, v)
    add = lambda *vs: None if any(v is None for v in vs) else sum(vs)
    for typ in range(8):
        au = tau if typ > 2 else 0
        for a in range(6):
            for b in range(6):
                em = ee = 0
                if typ:
                    if a < 5 and b < 5:
                        em, ee = clip(mm_m[(typ - 1) * 25 + a * 5 + b]), clip(mm_e[(typ - 1) * 25 + a * 5 + b])
                    elif a < 5:
                        em = ee = clip(d5[(typ - 1) * 5 + a])
                    elif b < 5:
                        em = ee = clip(d3[(typ - 1) * 5 + b])
                out += [add(em, au, ml["MLintern"]), add(ee, au)]
                if a < 5 and b < 5:
                    out.append(add(em, au, ml["MLintern"], ml["MLclosing"]))
    interior5 = flat(t, "interior")[5]
    out += [flat(t, "bulge")[1], add(interior5, m), ml["MLbase"]] + [min(mx, k * m) for k in range(1, 5)]
    return out


def mfe3_accepts(t):
    """mfe3.cu, mfe3_upload_tables: every asymmetry >= 5 capped (5 * ninio >= max_ninio), 0 <= max_ninio < 2000, and
    every int16 entry within +-TABLE_ENV16 = 2000 (INF entries do not fit: (short) of 10^7 wraps to -27008)"""
    m, mx = t.ninio()
    return m >= 0 and 5 * m >= mx and 0 <= mx < 2000 and all(v is not None and abs(v) <= 2000 for v in _int16_entries(t))


def mfe4_accepts(t):
    """mfe4.cu, mfe4_upload_tables (fits10): interior / 1xn mismatches and TerminalAU fit the 10-bit fields [-512, 512)"""
    vals = flat(t, "mismatch_interior")[:175] + flat(t, "mismatch_interior_1n")[:175] + [t.blocks["Misc"][0][2]]
    return all(v is not None and -MFE4_FIELD <= v < MFE4_FIELD for v in vals)


# ---- sequences
COMP = {"A": "U", "C": "G", "G": "C", "U": "A"}


def plant_special(t, rng, W, n_per_key=3):
    """sequences of length W, each with one special-loop key of `t` as the hairpin of a stem of up to 5 bp (the key's
    closing pair plus up to 4 more) in a random background: at the 5' edge, the 3' edge and an interior position"""
    out = []
    for key in t.special_keys():
        stem = min(4, (W - len(key)) // 2)
        if stem < 0:
            continue
        for where in range(n_per_key):
            s5 = "".join(rng.choice("GC") for _ in range(stem))
            motif = s5 + key + "".join(COMP[c] for c in reversed(s5))
            bg = [rng.choice("ACGU") for _ in range(W)]
            pos = (0, W - len(motif), rng.randrange(0, W - len(motif) + 1))[where % 3]
            bg[pos:pos + len(motif)] = motif
            out.append("".join(bg))
    return out
