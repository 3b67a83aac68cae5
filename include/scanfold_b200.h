/*
 * scanfold_b200.h -- C-ABI of the B200-native ScanFold scanning hot path (libscanfold_b200.so).
 *
 * The reference (moss-lab/ScanFold) has no FFI of its own: its hot path calls the ViennaRNA SWIG
 * module `RNA` once per fold from Python.  Each entry point below names the reference call sites it
 * replaces (file:line into /root/reference).  All functions return 0 on success or a negative SFB_E_*
 * code; sfb_last_error() gives the message.  The caller owns every buffer; inputs are never mutated.
 * Energies cross the boundary as int32 dcal (10 cal/mol), exactly ViennaRNA's internal unit; the Python
 * host converts with float32(e/100.) to mirror ScanFold.py:501.  There is NO CPU fallback in this library.
 */
#ifndef SCANFOLD_B200_H
#define SCANFOLD_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define SFB_VERSION 100
#define SFB_INF 10000000

#define SFB_E_ARG (-1)     /* bad argument */
#define SFB_E_PARAMS (-2)  /* parameter file missing / malformed */
#define SFB_E_CUDA (-3)    /* CUDA runtime error (no device, OOM, launch failure) */
#define SFB_E_STATE (-4)   /* sfb_init not called */
#define SFB_E_RANGE (-5)   /* window too long for this build */

#define SFB_SHUFFLE_MONO 0
#define SFB_SHUFFLE_DI 1

/* RNA.md(): only what the reference sets -- ScanFold.py:212-215, ScanFoldFunctions.py:776-777 */
typedef struct sfb_model {
    double temperature; /* md.temperature (C); tables are rescaled from the 37 C values and the enthalpies of the file */
    int32_t max_bp_span; /* md.max_bp_span; <=0 = unlimited */
} sfb_model;

int sfb_version(void);

/* Loads the energy tables (ViennaRNA "RNAfold parameter file v2.0"; NULL = built-in best-effort
 * Turner-2004 stand-in next to the library) and uploads them to device `device_ordinal`.
 * Replaces the implicit table load of `import RNA` (ScanFold.py:37). */
int sfb_init(int device_ordinal, const char *par_file_or_null);
void sfb_shutdown(void);
const char *sfb_last_error(void);
/* Launch everything on the caller's CUDA stream (a cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream)
 * so that the caller's events bracket the library's work; NULL = back to the library's own stream. */
int sfb_set_stream(void *cuda_stream_or_null);
/* Kernel selection for tests and tuning (results never depend on it): mfe_engine 1 = int32 CTA kernel (mfe.cu),
 * 2 = + int16 warp-team kernel (mfe2.cu), 3 = + int16 CTA kernel with stencil / range-minimum loops (mfe3.cu,
 * default); pf_engine 1 = global-memory kernel (pf.cu), 2 = + shared-memory kernel (pf2.cu, default).
 * A value <= 0 leaves that setting unchanged. */
int sfb_set_engines(int mfe_engine, int pf_engine);
/* 1 if the loaded table is the built-in best-effort stand-in (parity with ViennaRNA unpinned) */
int sfb_params_besteffort(void);

/* Batch of equal-length MFE folds.  Replaces RNA.fold_compound(seq, md).mfe():
 *   native window  ScanFold.py:494-497 / :512-513 (with hc) / :534-541 (with Deigan sc)
 *   background     ScanFoldFunctions.py:774-789 (rna_folder) via energies() :805-814
 * seqs  [n_seq*len] ASCII (ACGUT any case, others = N)
 * hc    NULL or [n_seq*len] constraint chars ". x | < > ( )"  (fc.hc_add_from_db, ScanFold.py:512)
 * sc    NULL or [n_seq*(len+1)] int32, 1-based per fold: stacking pseudo-energies in dcal
 *       (vrna_sc_add_SHAPE_deigan output, ScanFold.py:534)
 * e_dcal    [n_seq] out
 * pair_tbl  NULL (energy only) or [n_seq*len] int16 out: 1-based partner within the fold, 0 = unpaired */
int sfb_fold_batch(const uint8_t *seqs, int n_seq, int len, const sfb_model *model, const uint8_t *hc,
                   const int32_t *sc, int32_t *e_dcal, int16_t *pair_tbl);

/* One fold of a whole sequence, up to SFB_MAX_LONG nt, on the blocked int32 kernel (mfe4.cu).  Replaces the three full-length
 * folds of --global_refold: RNA.fold_compound(full sequence, md) [+ fc.hc_add_from_db(line 3 of a Zavg dbn file)] .mfe()
 * (ScanFold.py:1518-1539).  hc as in sfb_fold_batch (NULL = unconstrained).  pair_tbl [n] int32 out: 1-based partner,
 * 0 = unpaired (32-bit because a record can be longer than an int16 holds). */
#define SFB_MAX_LONG 40000
int sfb_fold_long(const uint8_t *seq, int n, const sfb_model *model, const uint8_t *hc, int32_t *e_dcal, int32_t *pair_tbl);

/* Batch of partition functions.  Replaces fc.pf(); fc.centroid(); fc.mean_bp_distance():
 *   ScanFold.py:498,503-504 / :514,518-519 / :525-527.
 * ensemble_dG [n_seq] kcal/mol, ed [n_seq] (mean_bp_distance), centroid_tbl [n_seq*len] int16 pair table,
 * bpp NULL or [n_seq*len*len] doubles (row i, col j, i<j). sc as in sfb_fold_batch (NULL in the scan loop). */
int sfb_pf_batch(const uint8_t *seqs, int n_seq, int len, const sfb_model *model, const uint8_t *hc,
                 const int32_t *sc, double *ensemble_dG, double *ed, int16_t *centroid_tbl, double *bpp);

/* Convert reactivities to Deigan stacking pseudo-energies: es[i] = (int)roundf((m*ln(r+1)+b)*100), 0 if r<0.
 * react1 / es1 are 1-based with n+1 entries.  Replaces fc.sc_add_SHAPE_deigan (ScanFold.py:534,539). */
int sfb_deigan(const double *react1, int n, double m, double b, int32_t *es1);

/* One record, one shard of windows: the whole scan loop ScanFold.py:429-692 (+ final-window block :694-757). */
typedef struct sfb_scan_args {
    const uint8_t *seq;  /* [L] ASCII RNA (T already transcribed to U by the caller, ScanFold.py:282) */
    int32_t L, W, step, r;
    int32_t shuffle_type;          /* SFB_SHUFFLE_MONO / _DI (scramble(), ScanFoldFunctions.py:834-851) */
    uint64_t seed;                 /* Philox key for device shuffles */
    const uint8_t *parity_shuffles; /* NULL, or [(n_windows+final_window)*r*W] host shuffles of THIS shard
                                     * (parity mode); must stay valid until the run finished */
    sfb_model model;
    const uint8_t *hc;   /* NULL or [L] constraint chars (line 3 of --constraints, ScanFold.py:401-410) */
    const double *react; /* NULL or [L+1] 1-based reactivities (getShapeDataFromFile, ScanFold.py:218-262) */
    double shape_m, shape_b;
    int32_t first_window, n_windows; /* shard: window indices [first_window, first_window+n_windows) */
    int32_t final_window;            /* 1: also evaluate the extra final-window set (Q5) as slot n_windows */
    int32_t want_pf;                 /* 1: partition function / ED / centroid per window */
    double background_temperature;   /* md.temperature of the r + 1 background folds (rna_folder, ScanFoldFunctions.py:776-777);
                                      * 0 = the same as model.temperature.  They differ in the motif step, where the native
                                      * fold uses the default 37 C compound and energies() gets -t (ScanFold.py:1733,1748) */
} sfb_scan_args;

typedef struct sfb_scan_out { /* caller-allocated; n = n_windows (+1 if final_window) */
    int32_t *mfe_dcal;                  /* [n] native MFE with hc/sc                 ScanFold.py:497/513/541 */
    int32_t *native_unconstrained_dcal; /* [n] energy_list[0]                        ScanFoldFunctions.py:808 */
    int32_t *shuffle_dcal;              /* [n*r] energy_list[1:]                                           */
    int16_t *pair_tbl;                  /* [n*W]                                                           */
    int16_t *centroid_tbl;              /* [n*W] (want_pf)                           ScanFold.py:503       */
    double *ed;                         /* [n]   (want_pf)                           ScanFold.py:504       */
    double *ensemble_dG;                /* [n]   (want_pf)                                                 */
    uint8_t *shuffles_out;              /* NULL or [n*r*W] the shuffled sequences actually folded           */
} sfb_scan_out;

int sfb_scan(const sfb_scan_args *args, sfb_scan_out *out);

/* Device-resident variant used to separate kernel time from copies (bench `value` vs `e2e`):
 * create uploads inputs and allocates device outputs; run launches the kernels on the library stream
 * and returns the CUDA-event time of the whole run and of the MFE kernels alone; fetch copies results out. */
typedef struct sfb_scan_plan sfb_scan_plan;
int sfb_scan_plan_create(const sfb_scan_args *args, sfb_scan_plan **plan);
/* call before run when sfb_scan_out.shuffles_out will be requested at fetch time */
void sfb_scan_plan_keep_shuffles(sfb_scan_plan *plan);
int sfb_scan_plan_run(sfb_scan_plan *plan, float *ms_total, float *ms_mfe, int32_t *n_launches);
int sfb_scan_plan_fetch(sfb_scan_plan *plan, sfb_scan_out *out);
/* CUDA-event times of the last run by stage: ms[0] window gather + shuffles, ms[1] MFE kernels, ms[2] partition
 * function kernels, ms[3] everything else (copies, final-window slot).  bench.py's roofline blocks use them. */
int sfb_scan_plan_stage_ms(const sfb_scan_plan *plan, float ms[4]);
void sfb_scan_plan_destroy(sfb_scan_plan *plan);

/* ScanFold-Fold accumulation step: the per-window pair records of ScanFold.py:564-677 gathered per nucleotide
 * and summed per (nucleotide, partner) as ScanFold.py:1051-1139 does with Python lists.  Runs on the device.
 * A shard of windows [first_window, first_window + n_windows) touches the nucleotides (0-based)
 * [first_window*step, (first_window+n_windows-1)*step + W): the table has one row per such nucleotide and
 * 2W-1 partner-offset columns.  Per cell: the number of windows holding the pair, the lowest window index
 * (first seen: the reference's dict insertion order) and EXACT sums of the window values z, MFE, ED: each
 * value d = k/100 enters as A = rint(d*2^20), B = (d - A*2^-20)*2^59, so sum(d) == sumA*2^-20 + sumB*2^-59
 * exactly -- order independent, which makes the multi-GPU halo merge bit exact.
 * Inputs are host arrays of the shard: pair_tbl [n_windows*W], z100 = round(z*100), mfe_dcal, ed100 = round(ED*100).
 * A window whose pair-table row is negative leaves no records (the all-N short-circuit of ScanFold.py:486-492). */
typedef struct sfb_accum_args {
    int32_t L, W, step, first_window, n_windows;
    const int16_t *pair_tbl;
    const int32_t *z100;
    const int32_t *mfe_dcal;
    const int32_t *ed100;
} sfb_accum_args;
typedef struct sfb_partner_table sfb_partner_table; /* device resident */
int sfb_accumulate_begin(const sfb_accum_args *args, sfb_partner_table **table);
int sfb_accumulate_geometry(const sfb_partner_table *table, int32_t *nt0, int32_t *n_nt);
/* Halo exchange between neighbouring shards (multi-GPU): copy rows [row0, row0+n_rows) out to / merge them in
 * from DEVICE buffers (count [n_rows*(2W-1)] int32, first_seen likewise, sums [6][n_rows*(2W-1)] int64) that the
 * caller moves with NCCL.  Merge adds counts and sums and takes the minimum of first_seen. */
int sfb_accumulate_export(sfb_partner_table *table, int row0, int n_rows, int32_t *d_count, int32_t *d_first_seen,
                          int64_t *d_sums);
int sfb_accumulate_merge(sfb_partner_table *table, int row0, int n_rows, const int32_t *d_count,
                         const int32_t *d_first_seen, const int64_t *d_sums);
/* Compact rows [row0, row0+n_rows) to per-nucleotide partner lists; returns the number of entries. */
int sfb_accumulate_compact(sfb_partner_table *table, int row0, int n_rows, int64_t *n_entries);
/* nparts [n_rows] entries per nucleotide (in column order); partner = 1-based partner coordinate (== own: unpaired);
 * sums [6][n_entries] = zA zB mfeA mfeB edA edB. */
int sfb_accumulate_fetch(sfb_partner_table *table, int32_t *nparts, int32_t *partner, int32_t *count,
                         int32_t *first_seen, int64_t *sums);
int sfb_accumulate_launches(const sfb_partner_table *table);
void sfb_accumulate_free(sfb_partner_table *table);

/* Window-averaged base-pair probabilities (the local pair-probability view of RNAplfold -W W -L W at step 1), kept
 * from the partition functions the scan already computes.  No reference counterpart (an additive output).
 * p^w(i,j) is the base-pair probability of (i,j) in the partition function of regular window w: the one whose ED
 * the scan reports (hard constraints and max_bp_span apply, soft constraints do not; the final-window slot is not a
 * window here).  With n(i,j) / n(i) the numbers of regular windows of the record that hold both i and j / hold i:
 *   P(i,j) = sum_w p^w(i,j) / n(i,j),   paired(i) = sum_w sum_k p^w(i,k) / n(i).
 * A table covers the nucleotides (0-based) [first_window*step, (first_window+n_windows-1)*step + W) of a shard of
 * windows: one row each, W int64 columns (0: sum of paired_w(i); d >= 1: sum of p^w(i,i+d)).  Every probability
 * enters as llrint(p * 2^40), so the sums are exact: the same for any chunking, split of the scan into plans, and
 * number of GPUs.  A window adds its probabilities once, from the run whose dG and ED are finite (a window out of the
 * fp64 range adds them from its rescaled retry). */
typedef struct sfb_pairprob_table sfb_pairprob_table;
int sfb_pairprob_begin(int32_t L, int32_t W, int32_t step, int32_t first_window, int32_t n_windows,
                       sfb_pairprob_table **table);
/* Attach `table` to a plan before sfb_scan_plan_run: every run then adds the probabilities of the plan's regular
 * windows to it.  The plan must compute the partition function (want_pf = 1), have the table's record length, W and
 * step, and its windows must lie in the table's range.  The table must outlive the plan's runs. */
int sfb_scan_plan_pairprob(sfb_scan_plan *plan, sfb_pairprob_table *table);
/* Halo exchange between neighbouring shards (multi-GPU): copy rows [row0, row0+n_rows) out to / add them in from a
 * DEVICE buffer of n_rows*W int64 that the caller moves with NCCL. */
int sfb_pairprob_export(sfb_pairprob_table *table, int row0, int n_rows, int64_t *d_rows);
int sfb_pairprob_merge(sfb_pairprob_table *table, int row0, int n_rows, const int64_t *d_rows);
/* Reduce rows [row0, row0+n_rows) on the device: paired(i) per row (0 where no window holds i) and the pairs with
 * P(i,j) >= cutoff (> 0), sorted by i then j; returns their number. */
int sfb_pairprob_compact(sfb_pairprob_table *table, int row0, int n_rows, double cutoff, int64_t *n_pairs);
/* Results of the last compact: paired [n_rows], i / j [n_pairs] 1-based record coordinates, p [n_pairs] = P(i,j). */
int sfb_pairprob_fetch(sfb_pairprob_table *table, double *paired, int32_t *i, int32_t *j, double *p);
void sfb_pairprob_free(sfb_pairprob_table *table);

/* Roofline denominators measured on the current device (bench.py): SFB_MICROBENCH_ADDMIN = int32
 * add-min (VIADDMNMX) operations per second over all SMs; SFB_MICROBENCH_SMEM_LD32 = conflict-free
 * 32-bit shared-memory loads per second (x4 = bytes/s).  No reference counterpart. */
#define SFB_MICROBENCH_ADDMIN 0
#define SFB_MICROBENCH_SMEM_LD32 1
#define SFB_MICROBENCH_DFMA 2 /* fp64 fused multiply-adds per second (partition-function roofline) */
int sfb_microbench(int which, double *ops_per_s);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif
