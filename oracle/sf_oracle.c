/*
 * sf_oracle.c -- CPU ORACLE (plain C restatement).  TEST INFRASTRUCTURE ONLY -- see sf_oracle.h.
 *
 * PARITY UNPINNED (see header).  Restates what the reference obtains from ViennaRNA at
 *   ScanFold.py:212-215 (RNA.md: temperature, max_bp_span), :494 (fold_compound), :497/:513/:541 (mfe),
 *   :498/:514/:525 (pf), :503 (centroid), :504 (mean_bp_distance), :512 (hc_add_from_db),
 *   :534 (sc_add_SHAPE_deigan), ScanFoldFunctions.py:774-789 (rna_folder background folds).
 * Algorithm statements follow SURVEY.md Appendix A (ViennaRNA 2.4.x, md defaults: dangles=2,
 * special_hp=1, noLP=0, noGU=0, TURN=3, MAXLOOP=30).
 */
#include "sf_oracle.h"
#include <ctype.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>

#define INF SFO_INF
#define TURN 3
#define MAXLOOP 30
#define NBPAIRS 7
#define MIN2(a, b) ((a) < (b) ? (a) : (b))
#define MAX2(a, b) ((a) > (b) ? (a) : (b))
#define K0 273.15
#define GASCONST 1.98717

typedef struct {
    char seq[10];
    int e;
} special_loop;

typedef struct {
    int loaded;
    int stack[8][8];
    int hairpin[31], bulge[31], internal_loop[31];
    int mismatchI[8][5][5], mismatchH[8][5][5], mismatch1nI[8][5][5], mismatch23I[8][5][5];
    int mismatchM_raw[8][5][5], mismatchExt_raw[8][5][5]; /* as in file (PF smooths these) */
    int mismatchM[8][5][5], mismatchExt[8][5][5];         /* clipped <= 0 for MFE (A.2) */
    int dangle5_raw[8][5], dangle3_raw[8][5], dangle5[8][5], dangle3[8][5];
    int int11[8][8][5][5];
    int int21[8][8][5][5][5];
    int int22[8][8][5][5][5][5];
    int MLbase, MLclosing, MLintern, ninio, max_ninio, TerminalAU, DuplexInit;
    double lxc;
    special_loop tetra[64], tri[64], hexa[64];
    int n_tetra, n_tri, n_hexa;
} params_t;

static params_t P;
static char g_err[512];
static long long g_dense, g_useful;
static int g_par_gen = 0; /* bumped by every sfo_load_params: invalidates derived tables */

static void set_err(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}
const char *sfo_last_error(void) { return g_err; }
void sfo_counters(long long *dense, long long *useful) {
    *dense = g_dense;
    *useful = g_useful;
}

/* ------------------------------------------------------------------ parameter file (A.3) */
typedef struct {
    char **tok;
    int n, pos;
} toks_t;

static char *read_all(const char *path) {
    FILE *f = fopen(path, "rb");
    if (!f) return NULL;
    fseek(f, 0, SEEK_END);
    long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    char *b = (char *)malloc(sz + 1);
    if (fread(b, 1, sz, f) != (size_t)sz) {
        fclose(f);
        free(b);
        return NULL;
    }
    b[sz] = 0;
    fclose(f);
    return b;
}

static void strip_comments(char *b) {
    for (char *p = b; *p; p++)
        if (p[0] == '/' && p[1] == '*') {
            char *q = strstr(p + 2, "*/");
            char *end = q ? q + 2 : p + strlen(p);
            for (char *r = p; r < end; r++)
                if (*r != '\n') *r = ' ';
            p = end - 1;
        }
}

static int tok_int(toks_t *t, int *ok) {
    if (t->pos >= t->n) {
        *ok = 0;
        return 0;
    }
    const char *s = t->tok[t->pos++];
    if (!strcmp(s, "INF")) return INF;
    if (!strcmp(s, "DEF")) return -50;
    char *e;
    long v = strtol(s, &e, 10);
    if (*e && *e != '.') *ok = 0;
    return (int)v;
}

static int read_ints(toks_t *t, int *dst, int count) {
    int ok = 1;
    for (int i = 0; i < count; i++) dst[i] = tok_int(t, &ok);
    return ok;
}

static int seek_block(toks_t *t, const char *name) {
    for (int i = 0; i + 1 < t->n; i++)
        if (!strcmp(t->tok[i], "#") && !strcmp(t->tok[i + 1], name)) {
            t->pos = i + 2;
            return 1;
        }
    return 0;
}

static int read_mm(toks_t *t, const char *name, int dst[8][5][5]) {
    if (!seek_block(t, name)) {
        set_err("missing block %s", name);
        return 0;
    }
    memset(dst, 0, sizeof(int) * 8 * 25);
    for (int ty = 1; ty <= 7; ty++)
        if (!read_ints(t, &dst[ty][0][0], 25)) {
            set_err("bad block %s", name);
            return 0;
        }
    return 1;
}

static int read_special(toks_t *t, const char *name, special_loop *dst, int *n) {
    *n = 0;
    if (!seek_block(t, name)) return 1; /* optional */
    while (t->pos + 2 < t->n + 1 && t->pos < t->n && isalpha((unsigned char)t->tok[t->pos][0]) &&
           strcmp(t->tok[t->pos], "INF")) {
        if (*n >= 64) break;
        strncpy(dst[*n].seq, t->tok[t->pos], 9);
        dst[*n].seq[9] = 0;
        dst[*n].e = atoi(t->tok[t->pos + 1]);
        t->pos += 3;
        (*n)++;
    }
    return 1;
}

/* one table set: suf "" = free energies at 37 C, "_enthalpies" = enthalpies; col 0 / 1 picks the value / its enthalpy in
 * the blocks that interleave them (ML_params, NINIO, Misc, special loops) */
static int read_special_col(toks_t *t, int col, const char *name, special_loop *dst, int *n) {
    *n = 0;
    if (!seek_block(t, name)) return 1; /* optional */
    while (t->pos + 2 < t->n + 1 && t->pos < t->n && isalpha((unsigned char)t->tok[t->pos][0]) &&
           strcmp(t->tok[t->pos], "INF")) {
        if (*n >= 64) break;
        strncpy(dst[*n].seq, t->tok[t->pos], 9);
        dst[*n].seq[9] = 0;
        dst[*n].e = atoi(t->tok[t->pos + 1 + col]);
        t->pos += 3;
        (*n)++;
    }
    return 1;
}

static int read_set(toks_t *t, const char *suf, int col, params_t *Q) {
    char nmbuf[8][64];
    int nmi = 0;
#define nm(x) (snprintf(nmbuf[nmi & 7], 64, "%s%s", x, suf), nmbuf[nmi++ & 7])
    memset(Q, 0, sizeof *Q);
    {
        if (!seek_block(t, nm("stack"))) {
            set_err("missing stack");
            return -1;
        }
        int ok = 1;
        for (int a = 1; a <= 7 && ok; a++) ok = read_ints(t, &Q->stack[a][1], 7);
        if (!ok) {
            set_err("bad stack");
            return -1;
        }
        if (!read_mm(t, nm("mismatch_hairpin"), Q->mismatchH)) return -1;
        if (!read_mm(t, nm("mismatch_interior"), Q->mismatchI)) return -1;
        if (!read_mm(t, nm("mismatch_interior_1n"), Q->mismatch1nI)) return -1;
        if (!read_mm(t, nm("mismatch_interior_23"), Q->mismatch23I)) return -1;
        if (!read_mm(t, nm("mismatch_multi"), Q->mismatchM_raw)) return -1;
        if (!read_mm(t, nm("mismatch_exterior"), Q->mismatchExt_raw)) return -1;
        if (!seek_block(t, nm("dangle5"))) {
            set_err("missing dangle5");
            return -1;
        }
        for (int a = 1; a <= 7 && ok; a++) ok = read_ints(t, &Q->dangle5_raw[a][0], 5);
        if (!seek_block(t, nm("dangle3"))) {
            set_err("missing dangle3");
            return -1;
        }
        for (int a = 1; a <= 7 && ok; a++) ok = read_ints(t, &Q->dangle3_raw[a][0], 5);
        if (!seek_block(t, nm("int11"))) {
            set_err("missing int11");
            return -1;
        }
        for (int a = 1; a <= 7 && ok; a++)
            for (int b = 1; b <= 7 && ok; b++) ok = read_ints(t, &Q->int11[a][b][0][0], 25);
        if (!seek_block(t, nm("int21"))) {
            set_err("missing int21");
            return -1;
        }
        for (int a = 1; a <= 7 && ok; a++)
            for (int b = 1; b <= 7 && ok; b++)
                for (int c = 0; c < 5 && ok; c++) ok = read_ints(t, &Q->int21[a][b][c][0][0], 25);
        if (!seek_block(t, nm("int22"))) {
            set_err("missing int22");
            return -1;
        }
        for (int a = 1; a <= 6 && ok; a++)
            for (int b = 1; b <= 6 && ok; b++)
                for (int c = 1; c <= 4 && ok; c++)
                    for (int d = 1; d <= 4 && ok; d++)
                        for (int e = 1; e <= 4 && ok; e++)
                            ok = read_ints(t, &Q->int22[a][b][c][d][e][1], 4);
        if (!ok) {
            set_err("bad int/dangle block");
            return -1;
        }
        if (!seek_block(t, nm("hairpin")) || !read_ints(t, Q->hairpin, 31)) {
            set_err("bad hairpin");
            return -1;
        }
        if (!seek_block(t, nm("bulge")) || !read_ints(t, Q->bulge, 31)) {
            set_err("bad bulge");
            return -1;
        }
        if (!seek_block(t, nm("interior")) || !read_ints(t, Q->internal_loop, 31)) {
            set_err("bad interior");
            return -1;
        }
        int ml[6], nin[3];
        if (!seek_block(t, "ML_params") || !read_ints(t, ml, 6)) {
            set_err("bad ML_params");
            return -1;
        }
        Q->MLbase = ml[0 + col];
        Q->MLclosing = ml[2 + col];
        Q->MLintern = ml[4 + col];
        if (!seek_block(t, "NINIO") || !read_ints(t, nin, 3)) {
            set_err("bad NINIO");
            return -1;
        }
        Q->ninio = nin[col];
        Q->max_ninio = nin[2];
        if (!seek_block(t, "Misc")) {
            set_err("missing Misc");
            return -1;
        }
        int misc[4];
        if (!read_ints(t, misc, 4)) {
            set_err("bad Misc");
            return -1;
        }
        Q->DuplexInit = misc[0 + col];
        Q->TerminalAU = misc[2 + col];
        Q->lxc = 107.856;
        if (t->pos < t->n && (isdigit((unsigned char)t->tok[t->pos][0]) || t->tok[t->pos][0] == '-'))
            Q->lxc = atof(t->tok[t->pos]);
        read_special_col(t, col, "Hexaloops", Q->hexa, &Q->n_hexa);
        read_special_col(t, col, "Tetraloops", Q->tetra, &Q->n_tetra);
        read_special_col(t, col, "Triloops", Q->tri, &Q->n_tri);
        /* int22 entries touching N (code 0): least favourable of the four nucleotides */
        for (int a = 1; a <= 6; a++)
            for (int b = 1; b <= 6; b++)
                for (int c = 0; c < 5; c++)
                    for (int d = 0; d < 5; d++)
                        for (int e = 0; e < 5; e++)
                            for (int f = 0; f < 5; f++) {
                                if (c && d && e && f) continue;
                                int m = -INF;
                                for (int c2 = (c ? c : 1); c2 <= (c ? c : 4); c2++)
                                    for (int d2 = (d ? d : 1); d2 <= (d ? d : 4); d2++)
                                        for (int e2 = (e ? e : 1); e2 <= (e ? e : 4); e2++)
                                            for (int f2 = (f ? f : 1); f2 <= (f ? f : 4); f2++)
                                                m = MAX2(m, Q->int22[a][b][c2][d2][e2][f2]);
                                Q->int22[a][b][c][d][e][f] = m;
                            }
    }
#undef nm
    return 0;
}

static params_t P37, PdH; /* what the file holds; P is the working set at g_temperature */
static double g_temperature = 37.0;

/* ViennaRNA get_scaled_params (md.temperature): E(T) = dH - (dH - E37) * (T + K0) / (37 + K0), truncated to int */
static void rescale_params(double T) {
    const int at37 = fabs(T - 37.0) < 1e-9;
    const double tempf = (T + K0) / (37.0 + K0);
    P = P37;
#define RS(field)                                                                                         \
    do {                                                                                                  \
        int *d = (int *)&P.field;                                                                         \
        const int *g = (const int *)&P37.field, *h = (const int *)&PdH.field;                             \
        for (size_t k = 0; k < sizeof(P.field) / sizeof(int); k++)                                        \
            d[k] = g[k] >= INF ? INF : (at37 ? g[k] : (int)((double)h[k] - (double)(h[k] - g[k]) * tempf)); \
    } while (0)
    RS(stack);
    RS(hairpin);
    RS(bulge);
    RS(internal_loop);
    RS(mismatchI);
    RS(mismatchH);
    RS(mismatch1nI);
    RS(mismatch23I);
    RS(mismatchM_raw);
    RS(mismatchExt_raw);
    RS(dangle5_raw);
    RS(dangle3_raw);
    RS(int11);
    RS(int21);
    RS(int22);
    RS(MLbase);
    RS(MLclosing);
    RS(MLintern);
    RS(ninio);
    RS(TerminalAU);
    RS(DuplexInit);
#undef RS
    for (int k = 0; k < 64; k++) {
        if (k < P.n_tetra) P.tetra[k].e = at37 ? P37.tetra[k].e : (int)((double)PdH.tetra[k].e - (double)(PdH.tetra[k].e - P37.tetra[k].e) * tempf);
        if (k < P.n_tri) P.tri[k].e = at37 ? P37.tri[k].e : (int)((double)PdH.tri[k].e - (double)(PdH.tri[k].e - P37.tri[k].e) * tempf);
        if (k < P.n_hexa) P.hexa[k].e = at37 ? P37.hexa[k].e : (int)((double)PdH.hexa[k].e - (double)(PdH.hexa[k].e - P37.hexa[k].e) * tempf);
    }
    P.max_ninio = P37.max_ninio;
    P.lxc = at37 ? P37.lxc : P37.lxc * tempf;
    /* MFE clips multi/exterior mismatches and dangles to <= 0 (A.2) */
    for (int a = 0; a < 8; a++)
        for (int b = 0; b < 5; b++) {
            P.dangle5[a][b] = MIN2(0, P.dangle5_raw[a][b]);
            P.dangle3[a][b] = MIN2(0, P.dangle3_raw[a][b]);
            for (int c = 0; c < 5; c++) {
                P.mismatchM[a][b][c] = MIN2(0, P.mismatchM_raw[a][b][c]);
                P.mismatchExt[a][b][c] = MIN2(0, P.mismatchExt_raw[a][b][c]);
            }
        }
    P.loaded = 1;
    g_temperature = T;
    g_par_gen++;
}

int sfo_set_temperature(double temperature_c) {
    if (!P37.loaded) {
        set_err("parameters not loaded");
        return -1;
    }
    if (temperature_c != g_temperature) rescale_params(temperature_c);
    return 0;
}

int sfo_load_params(const char *path) {
    char *buf = read_all(path);
    if (!buf) {
        set_err("cannot read %s", path);
        return -1;
    }
    if (strncmp(buf, "## RNAfold parameter file v2.0", 30)) {
        set_err("%s: not a v2.0 RNAfold parameter file", path);
        free(buf);
        return -1;
    }
    strip_comments(buf);
    /* tokenise; '#' becomes its own token so "# stack" -> "#","stack" ("#END" too) */
    toks_t t = {0};
    int cap = 1 << 16;
    t.tok = (char **)malloc(sizeof(char *) * cap);
    static char hash[] = "#";
    for (char *p = buf; *p;) {
        while (*p && isspace((unsigned char)*p)) p++;
        if (!*p) break;
        if (t.n + 2 >= cap) {
            cap *= 2;
            t.tok = (char **)realloc(t.tok, sizeof(char *) * cap);
        }
        if (*p == '#') {
            while (*p == '#') p++;
            t.tok[t.n++] = hash;
            continue;
        }
        t.tok[t.n++] = p;
        while (*p && !isspace((unsigned char)*p)) p++;
        if (*p) *p++ = 0;
    }
    int rc = -1;
    if (!read_set(&t, "", 0, &P37) && !read_set(&t, "_enthalpies", 1, &PdH)) {
        P37.loaded = PdH.loaded = 1;
        rescale_params(37.0);
        rc = 0;
    }
    free(t.tok);
    free(buf);
    return rc;
}

/* ------------------------------------------------------------------ encoding (A.1) */
static const int rtype[8] = {0, 2, 1, 4, 3, 6, 5, 7};
static int pair_tab[5][5];
static void init_pair_tab(void) {
    static int done = 0;
    if (done) return;
    memset(pair_tab, 0, sizeof pair_tab);
    pair_tab[2][3] = 1; /* CG */
    pair_tab[3][2] = 2; /* GC */
    pair_tab[3][4] = 3; /* GU */
    pair_tab[4][3] = 4; /* UG */
    pair_tab[1][4] = 5; /* AU */
    pair_tab[4][1] = 6; /* UA */
    done = 1;
}
static int enc(char c) {
    switch (toupper((unsigned char)c)) {
    case 'A': return 1;
    case 'C': return 2;
    case 'G': return 3;
    case 'U':
    case 'T': return 4;
    default: return 0;
    }
}

/* ------------------------------------------------------------------ loop energies (A.2) */
static int E_Hairpin(int u, int type, int si1, int sj1, const char *str /* points at s[i], upper-case RNA */) {
    int e = (u <= 30) ? P.hairpin[u] : P.hairpin[30] + (int)(P.lxc * log(u / 30.));
    if (u < 3) return e;
    if (u == 4)
        for (int k = 0; k < P.n_tetra; k++)
            if (!strncmp(str, P.tetra[k].seq, 6)) return P.tetra[k].e;
    if (u == 6)
        for (int k = 0; k < P.n_hexa; k++)
            if (!strncmp(str, P.hexa[k].seq, 8)) return P.hexa[k].e;
    if (u == 3) {
        for (int k = 0; k < P.n_tri; k++)
            if (!strncmp(str, P.tri[k].seq, 5)) return P.tri[k].e;
        return e + (type > 2 ? P.TerminalAU : 0);
    }
    return e + P.mismatchH[type][si1][sj1];
}

static int E_IntLoop(int n1, int n2, int type, int type_2, int si1, int sj1, int sp1, int sq1) {
    int nl, ns, e;
    if (n1 > n2) {
        nl = n1;
        ns = n2;
    } else {
        nl = n2;
        ns = n1;
    }
    if (nl == 0) return P.stack[type][type_2];
    if (ns == 0) {
        e = (nl <= MAXLOOP) ? P.bulge[nl] : P.bulge[30] + (int)(P.lxc * log(nl / 30.));
        if (nl == 1)
            e += P.stack[type][type_2];
        else {
            if (type > 2) e += P.TerminalAU;
            if (type_2 > 2) e += P.TerminalAU;
        }
        return e;
    }
    if (ns == 1) {
        if (nl == 1) return P.int11[type][type_2][si1][sj1];
        if (nl == 2) {
            if (n1 == 1) return P.int21[type][type_2][si1][sq1][sj1];
            return P.int21[type_2][type][sq1][si1][sp1];
        }
        e = (nl + 1 <= MAXLOOP) ? P.internal_loop[nl + 1]
                                : P.internal_loop[30] + (int)(P.lxc * log((nl + 1) / 30.));
        e += MIN2(P.max_ninio, (nl - ns) * P.ninio);
        e += P.mismatch1nI[type][si1][sj1] + P.mismatch1nI[type_2][sq1][sp1];
        return e;
    }
    if (ns == 2) {
        if (nl == 2) return P.int22[type][type_2][si1][sp1][sq1][sj1];
        if (nl == 3) {
            e = P.internal_loop[5] + P.ninio;
            e += P.mismatch23I[type][si1][sj1] + P.mismatch23I[type_2][sq1][sp1];
            return e;
        }
    }
    int u = nl + ns;
    e = (u <= MAXLOOP) ? P.internal_loop[u] : P.internal_loop[30] + (int)(P.lxc * log(u / 30.));
    e += MIN2(P.max_ninio, (nl - ns) * P.ninio);
    e += P.mismatchI[type][si1][sj1] + P.mismatchI[type_2][sq1][sp1];
    return e;
}

static int E_MLstem(int type, int si1, int sj1) {
    int e = 0;
    if (si1 >= 0 && sj1 >= 0)
        e += P.mismatchM[type][si1][sj1];
    else if (si1 >= 0)
        e += P.dangle5[type][si1];
    else if (sj1 >= 0)
        e += P.dangle3[type][sj1];
    if (type > 2) e += P.TerminalAU;
    return e + P.MLintern;
}

static int E_ExtLoop(int type, int si1, int sj1) {
    int e = 0;
    if (si1 >= 0 && sj1 >= 0)
        e += P.mismatchExt[type][si1][sj1];
    else if (si1 >= 0)
        e += P.dangle5[type][si1];
    else if (sj1 >= 0)
        e += P.dangle3[type][sj1];
    if (type > 2) e += P.TerminalAU;
    return e;
}

/* ------------------------------------------------------------------ fold context */
typedef struct {
    int n;
    char *s;          /* 1-based upper-case RNA string, s[0] unused, NUL at n+1 */
    int *S;           /* 1-based codes */
    unsigned char *ok; /* (n+2)*(n+2) pair permission (canonical, j-i>TURN, span, hc) -> type or 0 */
    const int *sc;    /* NULL or 1-based stacking pseudo-energies */
} ctx_t;

#define OK(c, i, j) ((c)->ok[(i) * ((c)->n + 2) + (j)])

/* hard constraints from a dot-bracket string with default options (A.5) */
static void apply_hc(ctx_t *c, const char *hc) {
    int n = c->n;
    int *stk = (int *)malloc(sizeof(int) * (n + 1)), sp = 0;
    int *mate = (int *)calloc(n + 2, sizeof(int));
    for (int i = 1; i <= n; i++) {
        char ch = hc[i - 1];
        if (ch == '(')
            stk[sp++] = i;
        else if (ch == ')') {
            if (sp > 0) {
                int k = stk[--sp];
                mate[k] = i;
                mate[i] = k;
            } /* unbalanced ')' ignored (Q8: version dependent) */
        }
    }
    free(stk); /* unmatched '(' ignored as well */
    for (int i = 1; i <= n; i++) {
        char ch = hc[i - 1];
        if (ch == 'x') {
            for (int k = 1; k <= n; k++) {
                OK(c, i, k) = 0;
                OK(c, k, i) = 0;
            }
        } else if (ch == '<') { /* may only pair downstream: forbid (k,i), k<i */
            for (int k = 1; k < i; k++) OK(c, k, i) = 0;
        } else if (ch == '>') { /* may only pair upstream: forbid (i,k), k>i */
            for (int k = i + 1; k <= n; k++) OK(c, i, k) = 0;
        } else if (ch == '(' && mate[i]) {
            int j = mate[i];
            /* weak enforcement: remove every pair conflicting with (i,j) */
            for (int p = 1; p <= n; p++)
                for (int q = p + 1; q <= n; q++) {
                    if (p == i && q == j) continue;
                    int conflict = (p == i || q == i || p == j || q == j) ||
                                   (p < i && i < q && q < j) || (i < p && p < j && j < q);
                    if (conflict) OK(c, p, q) = 0;
                }
        }
    }
    free(mate);
}

static int ctx_init(ctx_t *c, const char *seq, int n, const char *hc, const int *sc, int max_span) {
    init_pair_tab();
    if (!P.loaded) {
        set_err("parameters not loaded");
        return -1;
    }
    c->n = n;
    c->s = (char *)calloc(n + 3, 1);
    c->S = (int *)calloc(n + 3, sizeof(int));
    c->ok = (unsigned char *)calloc((size_t)(n + 2) * (n + 2), 1);
    c->sc = sc;
    for (int i = 1; i <= n; i++) {
        char ch = (char)toupper((unsigned char)seq[i - 1]);
        if (ch == 'T') ch = 'U';
        c->s[i] = ch;
        c->S[i] = enc(ch);
    }
    for (int i = 1; i <= n; i++)
        for (int j = i + TURN + 1; j <= n; j++) {
            if (max_span > 0 && j - i + 1 > max_span) continue;
            OK(c, i, j) = (unsigned char)pair_tab[c->S[i]][c->S[j]];
        }
    if (hc) apply_hc(c, hc);
    return 0;
}

static void ctx_free(ctx_t *c) {
    free(c->s);
    free(c->S);
    free(c->ok);
}

static int sc_stack4(const ctx_t *c, int i, int j, int p, int q) {
    if (!c->sc) return 0;
    return c->sc[i] + c->sc[p] + c->sc[q] + c->sc[j];
}

/* ------------------------------------------------------------------ MFE fill + traceback (A.4) */
typedef struct {
    int i, j, ml;
} sector_t;

static int mfe_core(ctx_t *c, char *structure, int count) {
    const int n = c->n;
    const int *S = c->S;
    const int N1 = n + 2;
    int *C = (int *)malloc(sizeof(int) * N1 * N1);
    int *M = (int *)malloc(sizeof(int) * N1 * N1);
    int *DM = (int *)malloc(sizeof(int) * N1 * N1); /* split-min of fML, the DMLi arrays */
    int *f5 = (int *)calloc(n + 2, sizeof(int));
#define CC(i, j) C[(i) * N1 + (j)]
#define MM(i, j) M[(i) * N1 + (j)]
#define DD(i, j) DM[(i) * N1 + (j)]
    for (int k = 0; k < N1 * N1; k++) C[k] = M[k] = DM[k] = INF;
    long long dense = 0, useful = 0;

    for (int i = n - TURN - 1; i >= 1; i--) {
        for (int j = i + TURN + 1; j <= n; j++) {
            int type = OK(c, i, j);
            if (type) {
                int new_c = E_Hairpin(j - i - 1, type, S[i + 1], S[j - 1], c->s + i);
                dense++;
                useful++;
                for (int p = i + 1; p <= MIN2(j - 2 - TURN, i + MAXLOOP + 1); p++) {
                    int minq = j - i + p - MAXLOOP - 2;
                    if (minq < p + 1 + TURN) minq = p + 1 + TURN;
                    for (int q = minq; q < j; q++) {
                        int t2 = OK(c, p, q);
                        if (!t2) continue;
                        t2 = rtype[t2];
                        int e = E_IntLoop(p - i - 1, j - q - 1, type, t2, S[i + 1], S[j - 1], S[p - 1], S[q + 1]);
                        if (p == i + 1 && q == j - 1) e += sc_stack4(c, i, j, p, q);
                        e += CC(p, q);
                        useful++;
                        if (e < new_c) new_c = e;
                    }
                }
                /* multiloop closed by (i,j): split-min of fML[i+1..j-1] */
                int d = DD(i + 1, j - 1);
                if (d < INF) {
                    int e = d + E_MLstem(rtype[type], S[j - 1], S[i + 1]) + P.MLclosing;
                    if (e < new_c) new_c = e;
                }
                CC(i, j) = new_c;
            }
            if (count) { /* dense relaxation count of SURVEY Appendix C (independent of pairability) */
                for (int p = i + 1; p <= MIN2(j - 2 - TURN, i + MAXLOOP + 1); p++) {
                    int minq = j - i + p - MAXLOOP - 2;
                    if (minq < p + 1 + TURN) minq = p + 1 + TURN;
                    if (j - 1 >= minq) dense += j - minq;
                }
                if (!type) dense++;
            }
            /* fML */
            int m = INF;
            if (MM(i + 1, j) < INF) m = MM(i + 1, j) + P.MLbase;
            if (MM(i, j - 1) < INF) m = MIN2(m, MM(i, j - 1) + P.MLbase);
            if (type && CC(i, j) < INF) {
                int e = CC(i, j) + E_MLstem(type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
                m = MIN2(m, e);
            }
            int dec = INF;
            for (int k = i + 1 + TURN; k <= j - 2 - TURN; k++) {
                dense++;
                if (MM(i, k) < INF && MM(k + 1, j) < INF) {
                    useful++;
                    int e = MM(i, k) + MM(k + 1, j);
                    if (e < dec) dec = e;
                }
            }
            DD(i, j) = dec;
            MM(i, j) = MIN2(m, dec);
        }
    }
    for (int j = 0; j <= MIN2(TURN + 1, n); j++) f5[j] = 0;
    for (int j = TURN + 2; j <= n; j++) {
        f5[j] = f5[j - 1];
        for (int i = j - TURN - 1; i >= 1; i--) {
            dense++;
            int type = OK(c, i, j);
            if (!type || CC(i, j) >= INF) continue;
            useful++;
            int e = f5[i - 1] + CC(i, j) + E_ExtLoop(type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
            if (e < f5[j]) f5[j] = e;
        }
    }
    int mfe = f5[n];
    if (count) {
        g_dense = dense;
        g_useful = useful;
    }

    if (structure) {
        int *pt = (int *)calloc(n + 2, sizeof(int));
        sector_t *stk = (sector_t *)malloc(sizeof(sector_t) * (2 * n + 8));
        int sp = 0, fail = 0;
        stk[sp].i = 1;
        stk[sp].j = n;
        stk[sp++].ml = 0;
        while (sp > 0 && !fail) {
            int i = stk[--sp].i, j = stk[sp].j, ml = stk[sp].ml;
            int have_pair = 0;
            if (ml == 2) {
                have_pair = 1;
            } else {
                if (j < i + TURN + 1) continue;
                int fij = ml ? MM(i, j) : f5[j];
                int fi = ml ? (MM(i, j - 1) < INF ? MM(i, j - 1) + P.MLbase : INF) : f5[j - 1];
                if (fij == fi) { /* 3' end unpaired */
                    stk[sp].i = i;
                    stk[sp].j = j - 1;
                    stk[sp++].ml = ml;
                    continue;
                }
                if (ml == 0) {
                    int k, found = 0;
                    for (k = j - TURN - 1; k >= 1; k--) {
                        int type = OK(c, k, j);
                        if (!type || CC(k, j) >= INF) continue;
                        if (fij == E_ExtLoop(type, k > 1 ? S[k - 1] : -1, j < n ? S[j + 1] : -1) + CC(k, j) + f5[k - 1]) {
                            found = 1;
                            break;
                        }
                    }
                    if (!found) {
                        fail = 1;
                        break;
                    }
                    stk[sp].i = 1;
                    stk[sp].j = k - 1;
                    stk[sp++].ml = 0;
                    i = k;
                    have_pair = 1;
                } else {
                    if (MM(i + 1, j) < INF && MM(i + 1, j) + P.MLbase == fij) { /* 5' end unpaired */
                        stk[sp].i = i + 1;
                        stk[sp].j = j;
                        stk[sp++].ml = 1;
                        continue;
                    }
                    int type = OK(c, i, j);
                    if (type && CC(i, j) < INF &&
                        fij == CC(i, j) + E_MLstem(type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1)) {
                        have_pair = 1;
                    } else {
                        int k;
                        for (k = i + 1 + TURN; k <= j - 2 - TURN; k++)
                            if (MM(i, k) < INF && MM(k + 1, j) < INF && fij == MM(i, k) + MM(k + 1, j)) break;
                        if (k > j - 2 - TURN) {
                            fail = 1;
                            break;
                        }
                        stk[sp].i = i;
                        stk[sp].j = k;
                        stk[sp++].ml = 1;
                        stk[sp].i = k + 1;
                        stk[sp].j = j;
                        stk[sp++].ml = 1;
                        continue;
                    }
                }
            }
            /* repeat1: (i,j) is a pair; descend through stacked / interior loops */
            while (have_pair) {
                pt[i] = j;
                pt[j] = i;
                int type = OK(c, i, j);
                int cij = CC(i, j);
                if (cij == E_Hairpin(j - i - 1, type, S[i + 1], S[j - 1], c->s + i)) break;
                int traced = 0;
                for (int p = i + 1; p <= MIN2(j - 2 - TURN, i + MAXLOOP + 1) && !traced; p++) {
                    int minq = j - i + p - MAXLOOP - 2;
                    if (minq < p + 1 + TURN) minq = p + 1 + TURN;
                    for (int q = j - 1; q >= minq; q--) {
                        int t2 = OK(c, p, q);
                        if (!t2 || CC(p, q) >= INF) continue;
                        t2 = rtype[t2];
                        int e = E_IntLoop(p - i - 1, j - q - 1, type, t2, S[i + 1], S[j - 1], S[p - 1], S[q + 1]);
                        if (p == i + 1 && q == j - 1) e += sc_stack4(c, i, j, p, q);
                        if (cij == e + CC(p, q)) {
                            i = p;
                            j = q;
                            traced = 1;
                            break;
                        }
                    }
                }
                if (traced) continue;
                /* multiloop */
                int en = cij - E_MLstem(rtype[type], S[j - 1], S[i + 1]) - P.MLclosing;
                int k;
                for (k = i + 2 + TURN; k < j - 2 - TURN; k++)
                    if (MM(i + 1, k) < INF && MM(k + 1, j - 1) < INF && en == MM(i + 1, k) + MM(k + 1, j - 1)) break;
                if (k <= j - 3 - TURN) {
                    stk[sp].i = i + 1;
                    stk[sp].j = k;
                    stk[sp++].ml = 1;
                    stk[sp].i = k + 1;
                    stk[sp].j = j - 1;
                    stk[sp++].ml = 1;
                } else
                    fail = 1;
                break;
            }
        }
        for (int i = 1; i <= n; i++) structure[i - 1] = pt[i] == 0 ? '.' : (pt[i] > i ? '(' : ')');
        structure[n] = 0;
        free(pt);
        free(stk);
        if (fail) {
            set_err("backtrack failed");
            mfe = INF;
        }
    }
    free(C);
    free(M);
    free(DM);
    free(f5);
    return mfe;
}

int sfo_mfe(const char *seq, int n, const char *hc, const int *sc_stack, int max_span, char *structure) {
    ctx_t c;
    if (ctx_init(&c, seq, n, hc, sc_stack, max_span)) return INF;
    int e = mfe_core(&c, structure, 1);
    ctx_free(&c);
    return e;
}

/* ------------------------------------------------------------------ independent structure evaluator */
int sfo_eval(const char *seq, int n, const char *structure, const int *sc_stack) {
    ctx_t c;
    if (ctx_init(&c, seq, n, NULL, sc_stack, 0)) return INF;
    int *pt = (int *)calloc(n + 2, sizeof(int));
    int *stk = (int *)malloc(sizeof(int) * (n + 1)), sp = 0;
    for (int i = 1; i <= n; i++) {
        if (structure[i - 1] == '(')
            stk[sp++] = i;
        else if (structure[i - 1] == ')') {
            if (!sp) {
                free(pt);
                free(stk);
                ctx_free(&c);
                return INF;
            }
            int k = stk[--sp];
            pt[k] = i;
            pt[i] = k;
        }
    }
    free(stk);
    const int *S = c.S;
    int e = 0;
    /* exterior loop */
    for (int i = 1; i <= n; i++)
        if (pt[i] > i) {
            int j = pt[i];
            int type = pair_tab[S[i]][S[j]];
            if (!type) type = 7;
            e += E_ExtLoop(type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
            i = j;
        }
    /* every pair closes one loop */
    for (int i = 1; i <= n; i++) {
        if (pt[i] <= i) continue;
        int j = pt[i];
        int type = pair_tab[S[i]][S[j]];
        if (!type) type = 7;
        int p = i + 1, nstem = 0, fp = 0, fq = 0;
        while (p < j) {
            if (pt[p] > p) {
                if (!nstem) {
                    fp = p;
                    fq = pt[p];
                }
                nstem++;
                p = pt[p] + 1;
            } else
                p++;
        }
        if (nstem == 0)
            e += E_Hairpin(j - i - 1, type, S[i + 1], S[j - 1], c.s + i);
        else if (nstem == 1) {
            int t2 = pair_tab[S[fp]][S[fq]];
            if (!t2) t2 = 7;
            e += E_IntLoop(fp - i - 1, j - fq - 1, type, rtype[t2], S[i + 1], S[j - 1], S[fp - 1], S[fq + 1]);
            if (fp == i + 1 && fq == j - 1) e += sc_stack4(&c, i, j, fp, fq);
        } else {
            e += P.MLclosing + E_MLstem(rtype[type], S[j - 1], S[i + 1]);
            int unp = j - i - 1;
            p = i + 1;
            while (p < j) {
                if (pt[p] > p) {
                    int q = pt[p];
                    int t2 = pair_tab[S[p]][S[q]];
                    if (!t2) t2 = 7;
                    e += E_MLstem(t2, S[p - 1], S[q + 1]);
                    unp -= q - p + 1;
                    p = q + 1;
                } else
                    p++;
            }
            e += unp * P.MLbase;
        }
    }
    free(pt);
    ctx_free(&c);
    return e;
}

/* ------------------------------------------------------------------ Deigan (A.6) */
void sfo_deigan(const double *react1, int n, double m, double b, int *es1) {
    es1[0] = 0;
    for (int i = 1; i <= n; i++) {
        double v = react1[i] < 0 ? 0. : m * log(react1[i] + 1) + b;
        es1[i] = (int)roundf((float)(v * 100.));
    }
}

/* ------------------------------------------------------------------ partition function (A.7) */
typedef struct pfpar_s {
    double kT, pf_scale;
    double expstack[8][8], exphairpin[31], expbulge[31], expinternal[31];
    double expmismatchI[8][5][5], expmismatchH[8][5][5], expmismatch1nI[8][5][5], expmismatch23I[8][5][5];
    double expmismatchM[8][5][5], expmismatchExt[8][5][5], expdangle5[8][5], expdangle3[8][5];
    double *expint11, *expint21, *expint22; /* same shapes as the int tables */
    double expMLbase, expMLclosing, expMLintern, expTermAU, expninio[MAXLOOP + 1];
    double exptetra[64], exptri[64], exphexa[64];
    double lxc;
} pfpar_t;

static double smooth(double X) { /* X in dcal (A.7) */
    double x = X / 10.;
    if (x < -1.2283697) return 0;
    if (x > 0.8660254) return X;
    double s = sin(x - 0.34242663) + 1;
    return 10. * 0.38490018 * s * s;
}

/* Boltzmann factors are a function of (parameter file, T): built once and kept (41 k exp() calls otherwise dominate
 * short windows); rebuilt when either changes.  Entries are never freed while a batch may still read them. */
static pthread_mutex_t g_pf_mu = PTHREAD_MUTEX_INITIALIZER;
static struct pfpar_s *g_pf_cache = NULL;
static double g_pf_cache_T = -1e9;
static int g_pf_cache_gen = -1;
static struct pfpar_s *pf_params_build(double T);
static struct pfpar_s *pf_params(double T) {
    pthread_mutex_lock(&g_pf_mu);
    if (!g_pf_cache || g_pf_cache_T != T || g_pf_cache_gen != g_par_gen) {
        g_pf_cache = pf_params_build(T);   /* the previous table set is leaked on purpose (rare: tests reload parameters) */
        g_pf_cache_T = T;
        g_pf_cache_gen = g_par_gen;
    }
    struct pfpar_s *q = g_pf_cache;
    pthread_mutex_unlock(&g_pf_mu);
    return q;
}
static struct pfpar_s *pf_params_build(double T) {
    pfpar_t *q = (pfpar_t *)calloc(1, sizeof(pfpar_t));
    double kT = (T + K0) * GASCONST; /* cal/mol */
    q->kT = kT;
#define BF(E) ((E) >= INF ? 0. : exp(-(double)(E) * 10. / kT))
    q->pf_scale = exp(-(-185 + (T - 37.) * 7.27) / kT);
    if (q->pf_scale < 1) q->pf_scale = 1;
    q->lxc = P.lxc;
    for (int i = 0; i <= 30; i++) {
        q->exphairpin[i] = BF(P.hairpin[i]);
        q->expbulge[i] = BF(P.bulge[i]);
        q->expinternal[i] = BF(P.internal_loop[i]);
    }
    for (int i = 0; i <= MAXLOOP; i++) q->expninio[i] = BF(MIN2(P.max_ninio, i * P.ninio));
    q->expMLbase = BF(P.MLbase);
    q->expMLclosing = BF(P.MLclosing);
    q->expMLintern = BF(P.MLintern);
    q->expTermAU = BF(P.TerminalAU);
    for (int k = 0; k < P.n_tetra; k++) q->exptetra[k] = BF(P.tetra[k].e);
    for (int k = 0; k < P.n_tri; k++) q->exptri[k] = BF(P.tri[k].e);
    for (int k = 0; k < P.n_hexa; k++) q->exphexa[k] = BF(P.hexa[k].e);
    q->expint11 = (double *)malloc(sizeof(double) * 8 * 8 * 25);
    q->expint21 = (double *)malloc(sizeof(double) * 8 * 8 * 125);
    q->expint22 = (double *)malloc(sizeof(double) * 8 * 8 * 625);
    for (int a = 0; a < 8; a++)
        for (int b = 0; b < 8; b++) {
            q->expstack[a][b] = BF(P.stack[a][b]);
            for (int k = 0; k < 25; k++) q->expint11[(a * 8 + b) * 25 + k] = BF((&P.int11[a][b][0][0])[k]);
            for (int k = 0; k < 125; k++) q->expint21[(a * 8 + b) * 125 + k] = BF((&P.int21[a][b][0][0][0])[k]);
            for (int k = 0; k < 625; k++) q->expint22[(a * 8 + b) * 625 + k] = BF((&P.int22[a][b][0][0][0][0])[k]);
        }
    for (int a = 0; a < 8; a++)
        for (int b = 0; b < 5; b++) {
            q->expdangle5[a][b] = exp(smooth(-P.dangle5_raw[a][b]) * 10. / kT);
            q->expdangle3[a][b] = exp(smooth(-P.dangle3_raw[a][b]) * 10. / kT);
            for (int cc = 0; cc < 5; cc++) {
                q->expmismatchI[a][b][cc] = BF(P.mismatchI[a][b][cc]);
                q->expmismatchH[a][b][cc] = BF(P.mismatchH[a][b][cc]);
                q->expmismatch1nI[a][b][cc] = BF(P.mismatch1nI[a][b][cc]);
                q->expmismatch23I[a][b][cc] = BF(P.mismatch23I[a][b][cc]);
                q->expmismatchM[a][b][cc] = exp(smooth(-P.mismatchM_raw[a][b][cc]) * 10. / kT);
                q->expmismatchExt[a][b][cc] = exp(smooth(-P.mismatchExt_raw[a][b][cc]) * 10. / kT);
            }
        }
    return q;
}
static void pf_params_free(pfpar_t *q) { (void)q; /* owned by the cache above */ }

static double exp_E_Hairpin(const pfpar_t *q, int u, int type, int si1, int sj1, const char *str) {
    double z = (u <= 30) ? q->exphairpin[u] : q->exphairpin[30] * exp(-(q->lxc * log(u / 30.)) * 10. / q->kT);
    if (u < 3) return z;
    if (u == 4)
        for (int k = 0; k < P.n_tetra; k++)
            if (!strncmp(str, P.tetra[k].seq, 6)) return q->exptetra[k];
    if (u == 6)
        for (int k = 0; k < P.n_hexa; k++)
            if (!strncmp(str, P.hexa[k].seq, 8)) return q->exphexa[k];
    if (u == 3) {
        for (int k = 0; k < P.n_tri; k++)
            if (!strncmp(str, P.tri[k].seq, 5)) return q->exptri[k];
        if (type > 2) z *= q->expTermAU;
        return z;
    }
    return z * q->expmismatchH[type][si1][sj1];
}

static double exp_E_IntLoop(const pfpar_t *q, int u1, int u2, int type, int type2, int si1, int sj1, int sp1, int sq1) {
    int ul = MAX2(u1, u2), us = MIN2(u1, u2);
    if (ul == 0) return q->expstack[type][type2];
    if (us == 0) {
        double z = q->expbulge[ul];
        if (ul == 1)
            z *= q->expstack[type][type2];
        else {
            if (type > 2) z *= q->expTermAU;
            if (type2 > 2) z *= q->expTermAU;
        }
        return z;
    }
    if (us == 1) {
        if (ul == 1) return q->expint11[((type * 8 + type2) * 5 + si1) * 5 + sj1];
        if (ul == 2) {
            if (u1 == 1) return q->expint21[(((type * 8 + type2) * 5 + si1) * 5 + sq1) * 5 + sj1];
            return q->expint21[(((type2 * 8 + type) * 5 + sq1) * 5 + si1) * 5 + sp1];
        }
        return q->expinternal[ul + us] * q->expmismatch1nI[type][si1][sj1] * q->expmismatch1nI[type2][sq1][sp1] *
               q->expninio[ul - us];
    }
    if (us == 2) {
        if (ul == 2) return q->expint22[((((type * 8 + type2) * 5 + si1) * 5 + sp1) * 5 + sq1) * 5 + sj1];
        if (ul == 3)
            return q->expinternal[5] * q->expmismatch23I[type][si1][sj1] * q->expmismatch23I[type2][sq1][sp1] *
                   q->expninio[1];
    }
    return q->expinternal[ul + us] * q->expmismatchI[type][si1][sj1] * q->expmismatchI[type2][sq1][sp1] *
           q->expninio[ul - us];
}

static double exp_E_MLstem(const pfpar_t *q, int type, int si1, int sj1) {
    double z = 1.;
    if (si1 >= 0 && sj1 >= 0)
        z = q->expmismatchM[type][si1][sj1];
    else if (si1 >= 0)
        z = q->expdangle5[type][si1];
    else if (sj1 >= 0)
        z = q->expdangle3[type][sj1];
    if (type > 2) z *= q->expTermAU;
    return z * q->expMLintern;
}
static double exp_E_ExtLoop(const pfpar_t *q, int type, int si1, int sj1) {
    double z = 1.;
    if (si1 >= 0 && sj1 >= 0)
        z = q->expmismatchExt[type][si1][sj1];
    else if (si1 >= 0)
        z = q->expdangle5[type][si1];
    else if (sj1 >= 0)
        z = q->expdangle3[type][sj1];
    if (type > 2) z *= q->expTermAU;
    return z;
}

static int pf_core(ctx_t *c, double T, double pf_scale, double *ensemble_dG, double *ed, char *centroid, double *bpp) {
    const int n = c->n, N1 = n + 2;
    const int *S = c->S;
    pfpar_t *pp = pf_params(T);
    const double ps = pf_scale > 0 ? pf_scale : pp->pf_scale;
    size_t sz = (size_t)N1 * N1;
    double *q = (double *)calloc(sz, sizeof(double)), *qb = (double *)calloc(sz, sizeof(double));
    double *qm = (double *)calloc(sz, sizeof(double)), *qm1 = (double *)calloc(sz, sizeof(double));
    double *pr = (double *)calloc(sz, sizeof(double));
    double *scale = (double *)malloc(sizeof(double) * (n + 3)), *eMLb = (double *)malloc(sizeof(double) * (n + 3));
#define Q(i, j) q[(i) * N1 + (j)]
#define QB(i, j) qb[(i) * N1 + (j)]
#define QM(i, j) qm[(i) * N1 + (j)]
#define QM1(i, j) qm1[(i) * N1 + (j)]
#define PR(i, j) pr[(i) * N1 + (j)]
    scale[0] = 1.;
    eMLb[0] = 1.;
    for (int i = 1; i <= n + 2; i++) {
        scale[i] = scale[i - 1] / ps;
        eMLb[i] = pow(pp->expMLbase, (double)i) * scale[i];
    }
    /* q[i][j] for j<i (empty) = 1; short segments = scale */
    for (int i = 1; i <= n + 1; i++) Q(i, i - 1) = 1.0;
    for (int d = 0; d <= TURN; d++)
        for (int i = 1; i + d <= n; i++) Q(i, i + d) = scale[d + 1];

    for (int j = TURN + 2; j <= n; j++) {
        for (int i = j - TURN - 1; i >= 1; i--) {
            int type = OK(c, i, j);
            double qbt1 = 0;
            if (type) {
                int u = j - i - 1;
                qbt1 = exp_E_Hairpin(pp, u, type, S[i + 1], S[j - 1], c->s + i) * scale[u + 2];
                for (int k = i + 1; k <= MIN2(i + MAXLOOP + 1, j - TURN - 2); k++) {
                    int u1 = k - i - 1;
                    for (int l = MAX2(k + TURN + 1, j - 1 - MAXLOOP + u1); l < j; l++) {
                        int t2 = OK(c, k, l);
                        if (!t2) continue;
                        t2 = rtype[t2];
                        double z = exp_E_IntLoop(pp, u1, j - l - 1, type, t2, S[i + 1], S[j - 1], S[k - 1], S[l + 1]);
                        if (c->sc && k == i + 1 && l == j - 1) z *= exp(-(double)sc_stack4(c, i, j, k, l) * 10. / pp->kT);
                        qbt1 += QB(k, l) * z * scale[u1 + j - l + 1];
                    }
                }
                double temp = 0;
                for (int k = i + 2; k <= j - 1; k++) temp += QM(i + 1, k - 1) * QM1(k, j - 1);
                qbt1 += temp * pp->expMLclosing * exp_E_MLstem(pp, rtype[type], S[j - 1], S[i + 1]) * scale[2];
            }
            QB(i, j) = qbt1;
            /* qm1[i,j]: exactly one stem starting at i, ending somewhere <= j */
            double v = QM1(i, j - 1) * eMLb[1];
            if (type) v += QB(i, j) * exp_E_MLstem(pp, type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
            QM1(i, j) = v;
            double temp = 0;
            for (int k = j; k > i; k--) temp += (QM(i, k - 1) + eMLb[k - i]) * QM1(k, j);
            QM(i, j) = temp + QM1(i, j);
        }
    }
    /* exterior: full q matrix (cubic, as in the library) */
    {
        double *qq = (double *)calloc(sz, sizeof(double)); /* qq[i][j]: stem i..j' ends exactly..: stems starting at i with 3' unpaired up to j */
#define QQ(i, j) qq[(i) * N1 + (j)]
        for (int j = TURN + 2; j <= n; j++)
            for (int i = j - TURN - 1; i >= 1; i--) {
                int type = OK(c, i, j);
                double qbt1 = QB(i, j);
                if (type) qbt1 *= exp_E_ExtLoop(pp, type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
                QQ(i, j) = QQ(i, j - 1) * scale[1] + qbt1;
                double temp = 1.0 * scale[1 + j - i] + QQ(i, j);
                for (int k = i; k <= j - 1; k++) temp += Q(i, k) * QQ(k + 1, j);
                Q(i, j) = temp;
            }
        free(qq);
    }
    double Z = Q(1, n);
    int out_of_range = !(Z > 0) || isinf(Z) || isnan(Z);
    if (ensemble_dG) *ensemble_dG = (-log(Z) - n * log(ps)) * pp->kT / 1000.0;

    /* outside: base pair probabilities */
    double *q1k = (double *)calloc(n + 3, sizeof(double)), *qln = (double *)calloc(n + 3, sizeof(double));
    for (int k = 1; k <= n; k++) {
        q1k[k] = Q(1, k);
        qln[k] = Q(k, n);
    }
    q1k[0] = 1.0;
    qln[n + 1] = 1.0;
    for (int i = 1; i <= n; i++)
        for (int j = i + TURN + 1; j <= n; j++) {
            int type = OK(c, i, j);
            if (type && QB(i, j) > 0.)
                PR(i, j) = q1k[i - 1] * qln[j + 1] / q1k[n] *
                           exp_E_ExtLoop(pp, type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
        }
    double *prml = (double *)calloc(n + 3, sizeof(double)), *prm_l = (double *)calloc(n + 3, sizeof(double));
    double *prm_l1 = (double *)calloc(n + 3, sizeof(double));
    for (int l = n; l > TURN + 1; l--) {
        /* (k,l) enclosed by (i,j) through an interior loop */
        for (int k = 1; k < l - TURN; k++) {
            int t2 = OK(c, k, l);
            if (!t2 || QB(k, l) == 0.) continue;
            t2 = rtype[t2];
            double tmp2 = 0;
            for (int i = MAX2(1, k - MAXLOOP - 1); i <= k - 1; i++)
                for (int j = l + 1; j <= MIN2(l + MAXLOOP - k + i + 2, n); j++) {
                    int type = OK(c, i, j);
                    if (type && PR(i, j) > 0) {
                        double z = exp_E_IntLoop(pp, k - i - 1, j - l - 1, type, t2, S[i + 1], S[j - 1], S[k - 1], S[l + 1]);
                        if (c->sc && k == i + 1 && l == j - 1) z *= exp(-(double)sc_stack4(c, i, j, k, l) * 10. / pp->kT);
                        tmp2 += PR(i, j) * scale[k - i + j - l] * z;
                    }
                }
            PR(k, l) += tmp2;
        }
        /* (k,l) as a stem of a multiloop closed by (i,j) */
        double prm_MLb = 0.;
        if (l < n)
            for (int k = 2; k < l - TURN; k++) {
                int i = k - 1;
                double prmt = 0, prmt1 = 0;
                int tt = OK(c, i, l + 1);
                if (tt) prmt1 = PR(i, l + 1) * pp->expMLclosing * exp_E_MLstem(pp, rtype[tt], S[l], S[i + 1]);
                for (int j = l + 2; j <= n; j++) {
                    tt = OK(c, i, j);
                    if (tt) prmt += PR(i, j) * exp_E_MLstem(pp, rtype[tt], S[j - 1], S[i + 1]) * QM(l + 1, j - 1);
                }
                prmt *= pp->expMLclosing;
                prml[i] = prmt;
                prm_l[i] = prm_l1[i] * eMLb[1] + prmt1;
                prm_MLb = prm_MLb * eMLb[1] + prml[i];
                prml[i] = prml[i] + prm_l[i];
                int tkl = OK(c, k, l);
                if (!tkl || QB(k, l) == 0.) continue;
                double temp = prm_MLb;
                for (int i2 = 1; i2 <= k - 2; i2++) temp += prml[i2] * QM(i2 + 1, k - 1);
                temp *= exp_E_MLstem(pp, tkl, k > 1 ? S[k - 1] : -1, l < n ? S[l + 1] : -1) * scale[2];
                PR(k, l) += temp;
            }
        double *tmp = prm_l1;
        prm_l1 = prm_l;
        prm_l = tmp;
    }
    double d = 0;
    int *pt = (int *)calloc(n + 2, sizeof(int));
    for (int i = 1; i <= n; i++)
        for (int j = i + TURN + 1; j <= n; j++) {
            double p = PR(i, j) * QB(i, j);
            PR(i, j) = p;
            d += p * (1 - p);
            if (p > 0.5) {
                pt[i] = j;
                pt[j] = i;
            }
            if (bpp) bpp[(size_t)(i - 1) * n + (j - 1)] = p;
        }
    if (ed) *ed = 2 * d;
    out_of_range |= isinf(d) || isnan(d);
    if (centroid) {
        for (int i = 1; i <= n; i++) centroid[i - 1] = pt[i] == 0 ? '.' : (pt[i] > i ? '(' : ')');
        centroid[n] = 0;
    }
    free(pt);
    free(prml);
    free(prm_l);
    free(prm_l1);
    free(q1k);
    free(qln);
    free(q);
    free(qb);
    free(qm);
    free(qm1);
    free(pr);
    free(scale);
    free(eMLb);
    pf_params_free(pp);
    if (out_of_range) set_err("pf overflow/underflow");
    return out_of_range ? 1 : 0;
}

int sfo_pf_scaled(const char *seq, int n, const char *hc, const int *sc_stack, int max_span, double temperature_c,
                  double pf_scale, double *ensemble_dG, double *ed, char *centroid, double *bpp) {
    ctx_t c;
    if (sfo_set_temperature(temperature_c)) return -1;
    if (ctx_init(&c, seq, n, hc, sc_stack, max_span)) return -1;
    if (bpp) memset(bpp, 0, sizeof(double) * (size_t)n * n);
    int rc = pf_core(&c, temperature_c, pf_scale, ensemble_dG, ed, centroid, bpp);
    ctx_free(&c);
    return rc ? -1 : 0;
}

int sfo_pf(const char *seq, int n, const char *hc, const int *sc_stack, int max_span, double temperature_c,
           double *ensemble_dG, double *ed, char *centroid, double *bpp) {
    int rc = sfo_pf_scaled(seq, n, hc, sc_stack, max_span, temperature_c, 0, ensemble_dG, ed, centroid, bpp);
    if (rc == 0) return 0;
    /* Z (or the outside pass) left the fp64 range under the fixed per-nucleotide scale: ViennaRNA's exp_params_rescale
     * rule, the scale from the MFE under the same constraints, pf_scale = exp(-1.07 mfe / (kT n)) */
    int e = sfo_mfe(seq, n, hc, sc_stack, max_span, NULL);
    if (e >= SFO_INF) return -1;
    double kT = (temperature_c + K0) * GASCONST;
    return sfo_pf_scaled(seq, n, hc, sc_stack, max_span, temperature_c, exp(-1.07 * e * 10. / (kT * n)), ensemble_dG, ed,
                         centroid, bpp);
}

/* Boltzmann weight (unscaled) of one structure under the PF energy model -- brute-force check of pf_core */
double sfo_eval_weight(const char *seq, int n, const char *structure, double T) {
    ctx_t c;
    if (ctx_init(&c, seq, n, NULL, NULL, 0)) return -1;
    pfpar_t *pp = pf_params(T);
    int *pt = (int *)calloc(n + 2, sizeof(int));
    int *stk = (int *)malloc(sizeof(int) * (n + 1)), sp = 0;
    for (int i = 1; i <= n; i++) {
        if (structure[i - 1] == '(')
            stk[sp++] = i;
        else if (structure[i - 1] == ')') {
            int k = stk[--sp];
            pt[k] = i;
            pt[i] = k;
        }
    }
    free(stk);
    const int *S = c.S;
    double w = 1.0;
    for (int i = 1; i <= n; i++)
        if (pt[i] > i) {
            int j = pt[i];
            w *= exp_E_ExtLoop(pp, pair_tab[S[i]][S[j]], i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
            i = j;
        }
    for (int i = 1; i <= n; i++) {
        if (pt[i] <= i) continue;
        int j = pt[i], type = pair_tab[S[i]][S[j]];
        int p = i + 1, nstem = 0, fp = 0, fq = 0;
        while (p < j) {
            if (pt[p] > p) {
                if (!nstem) {
                    fp = p;
                    fq = pt[p];
                }
                nstem++;
                p = pt[p] + 1;
            } else
                p++;
        }
        if (nstem == 0)
            w *= exp_E_Hairpin(pp, j - i - 1, type, S[i + 1], S[j - 1], c.s + i);
        else if (nstem == 1)
            w *= exp_E_IntLoop(pp, fp - i - 1, j - fq - 1, type, rtype[pair_tab[S[fp]][S[fq]]], S[i + 1], S[j - 1],
                               S[fp - 1], S[fq + 1]);
        else {
            w *= pp->expMLclosing * exp_E_MLstem(pp, rtype[type], S[j - 1], S[i + 1]);
            int unp = j - i - 1;
            p = i + 1;
            while (p < j) {
                if (pt[p] > p) {
                    int q = pt[p];
                    w *= exp_E_MLstem(pp, pair_tab[S[p]][S[q]], S[p - 1], S[q + 1]);
                    unp -= q - p + 1;
                    p = q + 1;
                } else
                    p++;
            }
            w *= pow(pp->expMLbase, unp);
        }
    }
    free(pt);
    pf_params_free(pp);
    ctx_free(&c);
    return w;
}

/* ------------------------------------------------------------------ batches (cpu_baseline) */
typedef struct {
    const char *seqs;
    int n_seq, len, mode;
    int *e;
    double *ed, *dG;
    char *cen;
    volatile int *next;
    int bad;
} job_t;

static void *worker(void *arg) {
    job_t *jb = (job_t *)arg;
    for (;;) {
        int k0 = __sync_fetch_and_add(jb->next, 4);
        if (k0 >= jb->n_seq) break;
        for (int k = k0; k < MIN2(k0 + 4, jb->n_seq); k++) {
            ctx_t c;
            ctx_init(&c, jb->seqs + (size_t)k * jb->len, jb->len, NULL, NULL, 0);
            if (jb->mode == 0)
                jb->e[k] = mfe_core(&c, NULL, 0);
            else if (pf_core(&c, 37.0, 0, jb->dG ? jb->dG + k : NULL, jb->ed + k,
                             jb->cen ? jb->cen + (size_t)k * (jb->len + 1) : NULL, NULL))
                jb->bad = 1;
            ctx_free(&c);
        }
    }
    return NULL;
}

static int run_batch(job_t *proto, int n_threads) {
    if (!P.loaded) {
        set_err("parameters not loaded");
        return -1;
    }
    init_pair_tab();
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    volatile int next = 0;
    job_t jobs[256];
    pthread_t th[256];
    for (int t = 0; t < n_threads; t++) {
        jobs[t] = *proto;
        jobs[t].next = &next;
        jobs[t].bad = 0;
        pthread_create(&th[t], NULL, worker, &jobs[t]);
    }
    int bad = 0;
    for (int t = 0; t < n_threads; t++) {
        pthread_join(th[t], NULL);
        bad |= jobs[t].bad;
    }
    return bad ? -1 : 0;
}

int sfo_fold_batch(const char *seqs, int n_seq, int len, int *e_dcal, int n_threads) {
    job_t jb = {seqs, n_seq, len, 0, e_dcal, NULL, NULL, NULL, NULL, 0};
    return run_batch(&jb, n_threads);
}

int sfo_pf_batch(const char *seqs, int n_seq, int len, double *ed, double *dG, char *centroids, int n_threads) {
    job_t jb = {seqs, n_seq, len, 1, NULL, ed, dG, centroids, NULL, 0};
    return run_batch(&jb, n_threads);
}

/* ------------------------------------------------------------------ fast batch path (bench CPU arm)
 * The same recursions as mfe_core for unconstrained, energy-only folds (the background folds of
 * ScanFoldFunctions.py:774-789 are > 99 % of a scan), written the way a tuned CPU library does it: one
 * reusable workspace per thread (no per-fold allocation or INF fill), the multiloop matrix kept in both
 * orientations so the split loop reads two contiguous rows, and the three separable interior-loop classes
 * (generic, 1xn, bulge) read copies of C that already carry the inner pair's mismatch term, so their inner
 * loops are branch-free add-min sweeps over contiguous memory that gcc vectorises.  The nine table-driven
 * shapes call E_IntLoop as before.  tests/test_oracle.py checks fast == simple fold by fold. */
typedef struct {
    int n;
    int *C, *G, *V1, *VB, *V1T, *VBT, *M, *MT, *DM, *f5, *S;
    unsigned char *T;
    char *s;
} fastws_t;

static void fastws_free(fastws_t *w) {
    free(w->C);
    free(w->f5);
    free(w->S);
    free(w->T);
    free(w->s);
    memset(w, 0, sizeof *w);
}

static int fastws_reserve(fastws_t *w, int n) {
    if (w->n >= n) return 0;
    fastws_free(w);
    const size_t N1 = (size_t)n + 2, sq = N1 * N1;
    w->C = (int *)malloc(sizeof(int) * sq * 9);
    w->f5 = (int *)malloc(sizeof(int) * (n + 2));
    w->S = (int *)malloc(sizeof(int) * (n + 3));
    w->T = (unsigned char *)malloc(sq);
    w->s = (char *)malloc(n + 3);
    if (!w->C || !w->f5 || !w->S || !w->T || !w->s) return -1;
    w->G = w->C + sq;
    w->V1 = w->G + sq;
    w->VB = w->V1 + sq;
    w->V1T = w->VB + sq;
    w->VBT = w->V1T + sq;
    w->M = w->VBT + sq;
    w->MT = w->M + sq;
    w->DM = w->MT + sq;
    w->n = n;
    return 0;
}

static int SZG[32][32];  /* generic loops: internal_loop[u1+u2] + asymmetry, reversed in u2: SZG[u1][30-u2] */
static int SZ1[32];      /* 1xn loops of total size u */
static int SZB[32];      /* bulges of size u */
static int g_fast_tables = 0;

static void fast_tables(void) {
    const int BIG = INF;
    for (int u1 = 0; u1 < 32; u1++)
        for (int k = 0; k < 32; k++) {
            const int u2 = 30 - k;
            int v = BIG;
            if (u1 >= 2 && u2 >= 2 && u1 + u2 <= MAXLOOP && !(u1 == 2 && u2 <= 3) && !(u2 == 2 && u1 <= 3))
                v = P.internal_loop[u1 + u2] + MIN2(P.max_ninio, abs(u1 - u2) * P.ninio);
            SZG[u1][k] = v;
        }
    for (int u = 0; u < 32; u++) {
        SZ1[u] = (u >= 4 && u <= MAXLOOP) ? P.internal_loop[u] + MIN2(P.max_ninio, (u - 2) * P.ninio) : BIG;
        SZB[u] = (u >= 2 && u <= MAXLOOP) ? P.bulge[u] : BIG;
    }
    g_fast_tables = 1;
}

static int mfe_fast(fastws_t *w, const char *seq, int n) {
    if (fastws_reserve(w, n)) return INF;
    const int N1 = n + 2;
    int *restrict C = w->C, *restrict G = w->G, *restrict V1 = w->V1, *restrict VB = w->VB;
    int *restrict V1T = w->V1T, *restrict VBT = w->VBT, *restrict M = w->M, *restrict MT = w->MT, *restrict DM = w->DM;
    unsigned char *restrict T = w->T;
    int *S = w->S;
    char *s = w->s;
    S[0] = S[n + 1] = S[n + 2] = 0;
    for (int i = 1; i <= n; i++) {
        char ch = (char)toupper((unsigned char)seq[i - 1]);
        if (ch == 'T') ch = 'U';
        s[i] = ch;
        S[i] = enc(ch);
    }
    s[0] = ' ';
    s[n + 1] = 0;
#define X(A, i, j) A[(i) * N1 + (j)]
    for (int i = n - TURN - 1; i >= 1; i--) {
        for (int j = i + TURN + 1; j <= n; j++) {
            const int type = pair_tab[S[i]][S[j]];
            X(T, i, j) = (unsigned char)type;
            int cij = INF;
            if (type) {
                const int si1 = S[i + 1], sj1 = S[j - 1];
                cij = E_Hairpin(j - i - 1, type, si1, sj1, s + i);
                /* the nine table-driven shapes */
                static const signed char SH[9][2] = {{0, 0}, {0, 1}, {1, 0}, {1, 1}, {1, 2}, {2, 1}, {2, 2}, {2, 3}, {3, 2}};
                for (int z = 0; z < 9; z++) {
                    const int p = i + 1 + SH[z][0], q = j - 1 - SH[z][1];
                    if (q - p <= TURN) continue;
                    const int t2 = X(T, p, q);
                    if (!t2) continue;
                    const int e = X(C, p, q) + E_IntLoop(SH[z][0], SH[z][1], type, rtype[t2], si1, sj1, S[p - 1], S[q + 1]);
                    if (e < cij) cij = e;
                }
                /* generic loops: rows p = i+1+u1, candidates contiguous in q */
                int bg = INF;
                for (int u1 = 2; u1 <= MAXLOOP - 2; u1++) {
                    const int p = i + 1 + u1;
                    int qlo = j - 1 - (MAXLOOP - u1), qhi = j - 3;
                    if (qlo < p + TURN + 1) qlo = p + TURN + 1;
                    if (qlo > qhi) {
                        if (p + TURN + 1 > qhi) break;
                        continue;
                    }
                    const int *restrict g = G + p * N1;
                    const int *restrict sz = SZG[u1] + (31 - j);   /* sz[q] = size term of u2 = j-1-q */
                    int b = INF;
                    for (int q = qlo; q <= qhi; q++) {
                        const int e = g[q] + sz[q];
                        b = e < b ? e : b;
                    }
                    bg = b < bg ? b : bg;
                }
                if (bg < INF) {
                    bg += P.mismatchI[type][si1][sj1];
                    if (bg < cij) cij = bg;
                }
                /* 1xn loops: u1 = 1 along row i+2, u2 = 1 along column j-2 (transposed copy) */
                {
                    int b = INF;
                    const int p = i + 2;
                    int qlo = j - 1 - (MAXLOOP - 1), qhi = j - 4;
                    if (qlo < p + TURN + 1) qlo = p + TURN + 1;
                    const int *restrict v = V1 + p * N1;
                    for (int q = qlo; q <= qhi; q++) {   /* total size u = 1 + (j-1-q) */
                        const int e = v[q] + SZ1[j - q];
                        b = e < b ? e : b;
                    }
                    const int q2 = j - 2;
                    int plo = i + 4, phi = i + 1 + (MAXLOOP - 1);
                    if (phi > q2 - TURN - 1) phi = q2 - TURN - 1;
                    const int *restrict vt = V1T + q2 * N1;
                    for (int pp = plo; pp <= phi; pp++) {   /* u = (pp-i-1) + 1 */
                        const int e = vt[pp] + SZ1[pp - i];
                        b = e < b ? e : b;
                    }
                    if (b < INF) {
                        b += P.mismatch1nI[type][si1][sj1];
                        if (b < cij) cij = b;
                    }
                }
                /* bulges of size >= 2 */
                {
                    int b = INF;
                    const int p = i + 1;
                    int qlo = j - 1 - MAXLOOP, qhi = j - 3;
                    if (qlo < p + TURN + 1) qlo = p + TURN + 1;
                    const int *restrict v = VB + p * N1;
                    for (int q = qlo; q <= qhi; q++) {
                        const int e = v[q] + SZB[j - 1 - q];
                        b = e < b ? e : b;
                    }
                    const int q2 = j - 1;
                    int plo = i + 3, phi = i + 1 + MAXLOOP;
                    if (phi > q2 - TURN - 1) phi = q2 - TURN - 1;
                    const int *restrict vt = VBT + q2 * N1;
                    for (int pp = plo; pp <= phi; pp++) {
                        const int e = vt[pp] + SZB[pp - i - 1];
                        b = e < b ? e : b;
                    }
                    if (b < INF) {
                        b += type > 2 ? P.TerminalAU : 0;
                        if (b < cij) cij = b;
                    }
                }
                /* multiloop closed by (i,j) */
                if (j - i - 2 > TURN) {
                    const int d = X(DM, i + 1, j - 1);
                    if (d < INF) {
                        const int e = d + E_MLstem(rtype[type], sj1, si1) + P.MLclosing;
                        if (e < cij) cij = e;
                    }
                }
            }
            X(C, i, j) = cij;
            {
                int vg = INF, v1 = INF, vb = INF;
                if (type && i > 1 && j < n) {
                    const int t2 = rtype[type];
                    vg = cij + P.mismatchI[t2][S[j + 1]][S[i - 1]];
                    v1 = cij + P.mismatch1nI[t2][S[j + 1]][S[i - 1]];
                    vb = cij + (t2 > 2 ? P.TerminalAU : 0);
                }
                X(G, i, j) = vg;
                X(V1, i, j) = v1;
                X(VB, i, j) = vb;
                X(V1T, j, i) = v1;
                X(VBT, j, i) = vb;
            }
            /* fML */
            int m = INF;
            if (j - i - 1 > TURN) {
                const int a = X(M, i + 1, j), b = X(M, i, j - 1);
                if (a < INF) m = a + P.MLbase;
                if (b < INF && b + P.MLbase < m) m = b + P.MLbase;
            }
            if (type) {
                const int e = cij + E_MLstem(type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
                if (e < m) m = e;
            }
            int dec = 2 * INF;
            {
                const int *restrict a = M + i * N1;          /* M[i][k] */
                const int *restrict b = MT + j * N1 + 1;     /* MT[j][k+1] = M[k+1][j] */
                for (int k = i + 1 + TURN; k <= j - 2 - TURN; k++) {
                    const int e = a[k] + b[k];
                    dec = e < dec ? e : dec;
                }
            }
            if (dec >= INF - 1000000) dec = INF;
            X(DM, i, j) = dec;
            m = MIN2(m, dec);
            X(M, i, j) = m;
            X(MT, j, i) = m;
        }
    }
    int *f5 = w->f5;
    for (int j = 0; j <= MIN2(TURN + 1, n); j++) f5[j] = 0;
    for (int j = TURN + 2; j <= n; j++) {
        int best = f5[j - 1];
        for (int i = j - TURN - 1; i >= 1; i--) {
            const int type = X(T, i, j);
            if (!type) continue;
            const int e = f5[i - 1] + X(C, i, j) + E_ExtLoop(type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
            if (e < best) best = e;
        }
        f5[j] = best;
    }
#undef X
    return f5[n];
}

static void *worker_fast(void *arg) {
    job_t *jb = (job_t *)arg;
    fastws_t ws;
    memset(&ws, 0, sizeof ws);
    for (;;) {
        int k0 = __sync_fetch_and_add(jb->next, 8);
        if (k0 >= jb->n_seq) break;
        for (int k = k0; k < MIN2(k0 + 8, jb->n_seq); k++) {
            jb->e[k] = mfe_fast(&ws, jb->seqs + (size_t)k * jb->len, jb->len);
            if (jb->e[k] >= INF) jb->bad = 1;
        }
    }
    fastws_free(&ws);
    return NULL;
}

int sfo_fold_batch_fast(const char *seqs, int n_seq, int len, int *e_dcal, int n_threads) {
    if (!P.loaded) {
        set_err("parameters not loaded");
        return -1;
    }
    init_pair_tab();
    fast_tables();
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    volatile int next = 0;
    job_t jobs[256];
    pthread_t th[256];
    for (int t = 0; t < n_threads; t++) {
        job_t jb = {seqs, n_seq, len, 0, e_dcal, NULL, NULL, NULL, &next, 0};
        jobs[t] = jb;
        pthread_create(&th[t], NULL, worker_fast, &jobs[t]);
    }
    int bad = 0;
    for (int t = 0; t < n_threads; t++) {
        pthread_join(th[t], NULL);
        bad |= jobs[t].bad;
    }
    if (bad) set_err("fast fold failed");
    return bad ? -1 : 0;
}
