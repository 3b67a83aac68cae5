/*
 * sf_oracle.h -- CPU ORACLE for the ScanFold scanning hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this library.  The product (scanfold_b200/) never links, imports or calls it.
 *
 * PARITY UNPINNED: the reference (moss-lab/ScanFold) has no fold code and no tests; every energy
 * comes from the external ViennaRNA C library (ScanFold.py:37,494-544; ScanFoldFunctions.py:774-789)
 * which is absent from /root/reference and from this image.  This file restates the published
 * ViennaRNA 2.4.x algorithms (Zuker/Turner-2004 MFE with dangles=2, McCaskill partition function)
 * from memory (SURVEY.md Appendix A).  No ViennaRNA golden vector exists to pin it.
 */
#ifndef SF_ORACLE_H
#define SF_ORACLE_H
#ifdef __cplusplus
extern "C" {
#endif

#define SFO_INF 10000000

/* load a ViennaRNA "## RNAfold parameter file v2.0"; returns 0 on success */
int sfo_load_params(const char *path);
const char *sfo_last_error(void);
/* md.temperature (ScanFold.py:213, ScanFoldFunctions.py:777): rescale every table from the 37 C values and the enthalpy
 * blocks of the file, E(T) = dH - (dH - E37) (T + 273.15) / 310.15 truncated to int (SURVEY A.3).  Process-wide; the
 * batch functions use whatever was set last.  sfo_pf sets it from its own temperature argument. */
int sfo_set_temperature(double temperature_c);

/* RNA.fold_compound(seq, md).mfe()  -- ScanFold.py:494-497,513,541; ScanFoldFunctions.py:786-787.
 * seq: n chars (ACGUT, any case).  hc: NULL or n chars of ". x | < > ( )" (fc.hc_add_from_db, ScanFold.py:512).
 * sc_stack: NULL or n+1 ints (1-based, dcal) = Deigan stacking pseudo energies (ScanFold.py:534).
 * max_span <= 0 means unlimited (md.max_bp_span, ScanFold.py:215).
 * structure: n+1 chars out (NUL terminated) or NULL for energy only.   Returns energy in dcal. */
int sfo_mfe(const char *seq, int n, const char *hc, const int *sc_stack, int max_span,
            char *structure);

/* energy of a given structure under the same model (independent loop evaluator) */
int sfo_eval(const char *seq, int n, const char *structure, const int *sc_stack);

/* fc.pf(); fc.centroid(); fc.mean_bp_distance()  -- ScanFold.py:498-504,514-519,525-527.
 * bpp: NULL or n*n doubles (row i-1, col j-1, i<j).  Returns 0 on success. */
int sfo_pf(const char *seq, int n, const char *hc, const int *sc_stack, int max_span,
           double temperature_c, double *ensemble_dG, double *ed, char *centroid, double *bpp);
/* sfo_pf first uses the fixed per-nucleotide scale of the tables (ViennaRNA's default pf_scale); where Z or the outside
 * pass leaves the fp64 range it computes again with exp_params_rescale's scale exp(-1.07 mfe / (kT n)), mfe under the
 * same constraints.  sfo_pf_scaled uses `pf_scale` (> 0; 0 = the default) and returns -1 if the range is left. */
int sfo_pf_scaled(const char *seq, int n, const char *hc, const int *sc_stack, int max_span, double temperature_c,
                  double pf_scale, double *ensemble_dG, double *ed, char *centroid, double *bpp);

/* Boltzmann weight of one structure under the PF model (brute-force checks) */
double sfo_eval_weight(const char *seq, int n, const char *structure, double T);

/* vrna_sc_add_SHAPE_deigan conversion: reactivities[1..n] -> es[1..n] in dcal (SURVEY A.6) */
void sfo_deigan(const double *react1, int n, double m, double b, int *es1);

/* batch of equal-length folds, energy only, OpenMP over folds (bench cpu_baseline) */
int sfo_fold_batch(const char *seqs, int n_seq, int len, int *e_dcal, int n_threads);
/* the same energies through the tuned path (per-thread reusable buffers, vectorisable inner loops): what a CPU
 * library would run; bench.py's CPU arm times this one, tests check it against sfo_fold_batch fold by fold */
int sfo_fold_batch_fast(const char *seqs, int n_seq, int len, int *e_dcal, int n_threads);
/* batch of PF/ED (no constraints) */
int sfo_pf_batch(const char *seqs, int n_seq, int len, double *ed, double *dG, char *centroids,
                 int n_threads);

/* work counters (SURVEY 8d): dense and useful relaxations of the last sfo_mfe call */
void sfo_counters(long long *dense, long long *useful);

#ifdef __cplusplus
}
#endif
#endif
