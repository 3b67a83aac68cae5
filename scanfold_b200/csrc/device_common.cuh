// Shared device-side definitions for the fold kernels.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "params.hpp"

namespace sfb {

// pair type of two nucleotide codes (SURVEY A.1): CG=1 GC=2 GU=3 UG=4 AU=5 UA=6
__host__ __device__ __forceinline__ int pair_type(int a, int b) {
    // 5x5 table packed 3 bits per entry would not fit 64 bits; use arithmetic on the 6 canonical cases
    int k = a * 5 + b;
    return k == 13 ? 1 : k == 17 ? 2 : k == 19 ? 3 : k == 23 ? 4 : k == 9 ? 5 : k == 21 ? 6 : 0;
}
__host__ __device__ __forceinline__ int rtype_of(int t) {
    // {0,2,1,4,3,6,5,7}
    return t == 0 ? 0 : (t == 7 ? 7 : ((t - 1) ^ 1) + 1);
}

// triangular diagonal-major index: diagonal d (= j - i) holds W - d cells, cell i at tri(d) + i
__host__ __device__ __forceinline__ int tri_off(int d, int W) { return d * W - (d * (d - 1)) / 2; }

// Pair permission under the default hard-constraint rules of fc.hc_add_from_db (SURVEY A.5):
// canonical pair, j - i > TURN, max_bp_span, 'x' / '<' / '>' flags, weakly enforced '(' ')' pairs.
struct HcCtx {
    const uint8_t *S;     // nucleotide codes
    const uint8_t *hcf;   // per-base flags (1: 'x', 2: '<', 4: '>') or NULL
    const int16_t *mate;  // enforced partner (-1 none) or NULL
    int W, max_span, n_enf;
};

__device__ inline int allowed_type(const HcCtx &c, int i, int j) {
    int t = pair_type(c.S[i], c.S[j]);
    if (!t) return 0;
    int d = j - i;
    if (d <= TURN) return 0;
    if (c.max_span > 0 && d + 1 > c.max_span) return 0;
    if (c.hcf) {
        int fi = c.hcf[i], fj = c.hcf[j];
        if ((fi | fj) & 1) return 0;  // 'x'
        if (fj & 2) return 0;         // '<' : j may only pair downstream
        if (fi & 4) return 0;         // '>' : i may only pair upstream
        if (c.n_enf) {
            int mi = c.mate[i], mj = c.mate[j];
            if (mi >= 0 && mi != j) return 0;
            if (mj >= 0 && mj != i) return 0;
            if (mi != j) {
                for (int a = 0; a < c.W; a++) {
                    int b = c.mate[a];
                    if (b <= a) continue;
                    if ((a < i && i < b && b < j) || (i < a && a < j && j < b)) return 0;
                }
            }
        }
    }
    return t;
}

__device__ inline int loop_key_dev(const uint8_t *S, int i, int n) {
    int key = 0, mul = 1;
    for (int k = 0; k < n; k++) {
        key += S[i + k] * mul;
        mul *= 5;
    }
    return key;
}

struct MfeLaunch {
    const uint8_t *seqs;  // [n_fold][W] nucleotide codes 0..4
    const uint8_t *hc;    // NULL or [n_fold][W] constraint characters
    const int32_t *sc;    // NULL or [n_fold][W+1] 1-based stacking pseudo-energies (dcal)
    int n_fold, W, max_span;
    int32_t *e_out;       // [n_fold]
    int16_t *pair_tbl;    // NULL or [n_fold][W]
    int32_t *gscratch;    // global scratch for matrices that do not fit shared memory
    long long gscratch_per_cta;  // ints
    int mats_in_gmem;     // 0: everything in shared memory; 1: C/FML in global; 2: rolling buffers too
    int redo_only;        // 1: only folds whose e_out holds MFE_REDO (flagged by the int16 kernel)
    int hc_simple;        // hc holds no '(' ')' : per-nucleotide flags only ('x' '<' '>'), which mfe3 folds in
};
constexpr int MFE_REDO = 0x7fffff00;  // e_out marker: int16 range exceeded, fold again in int32

struct PfLaunch {
    const uint8_t *seqs;  // [n_fold][W] codes
    const uint8_t *hc;    // NULL or [n_fold][W]
    const int32_t *sc;    // NULL or [n_fold][W+1]
    int n_fold, W, max_span;
    double *dG, *ed;      // [n_fold]
    int16_t *centroid;    // [n_fold][W]
    double *bpp;          // NULL or [n_fold][W][W]
    double *gscratch;     // per-CTA workspace
    long long gscratch_per_cta;  // doubles
    int hc_simple;        // hc holds no '(' ')' : per-nucleotide flags only, which pf2 folds in
    double pf_scale;      // 0: the tables' per-nucleotide scale; > 0: this one (range retry, pf.cu only)
    int *n_out_of_range;  // NULL or a counter: +1 per fold whose dG or ED is not finite (Z left the fp64 range)
};
// Where a PF launch commits its probabilities (pairprob.cu), a kernel argument of its own so that the PfLaunch of the
// default path keeps its layout.  table NULL: none.  A fold whose dG and ED come out finite adds its probabilities to
// rows row0 + fold * step + i of the table (W columns each, see PairProbDense); a fold out of the fp64 range adds nothing.
struct PairProbCommit {
    long long *table;
    long long row0;
    int step;
};

void launch_mfe(const MfeLaunch &L, const MfeTables *d_tab, int n_sm, cudaStream_t stream, int *n_launches);
size_t mfe_scratch_ints_per_cta(int W, int *mats_in_gmem);
// second-generation energy-only kernel (mfe2.cu): one warp per fold, W <= 128, no constraints
bool mfe2_supports(int W);
int mfe2_grid_size(int n_sm, int n_fold);
size_t mfe2_scratch_shorts_per_warp(int W);
void mfe2_upload_tables(const MfeTables &M);
void launch_mfe2(const MfeLaunch &L, const MfeTables *d_tab, int n_sm, cudaStream_t stream, int *n_launches);
// third-generation energy-only kernel (mfe3.cu): one CTA per fold, stencil / range-minimum interior loops
bool mfe3_supports(int W);
int mfe3_max_ctas(int n_sm, int W);
size_t mfe3_scratch_shorts_per_cta(int W);
void mfe3_upload_tables(const MfeTables &M);
void launch_mfe3(const MfeLaunch &L, const MfeTables *d_tab, int n_sm, cudaStream_t stream, int *n_launches);
int mfe_grid_size(int W, int n_sm, int n_fold);
// fourth-generation kernel (mfe4.cu): blocked int32 fill in HBM for windows above 300 nt and whole-sequence folds.
// `scratch` holds the matrices of as many folds as fit (mfe4_bytes_per_fold each; at least one); d_hp_len = hairpin
// initiation by loop size [W + 1] on the device; pair32 = optional 32-bit pair table (whole-sequence folds)
void mfe4_upload_tables(const MfeTables &M);
bool mfe4_supports(int n);
size_t mfe4_bytes_per_fold(int n);
void launch_mfe4(const MfeLaunch &L, const MfeTables *d_tab, const int32_t *d_hp_len, void *scratch, size_t scratch_bytes,
                 int32_t *pair32, int n_sm, cudaStream_t stream, int *n_launches);

void launch_pf(const PfLaunch &L, const MfeTables *d_mfe, const PfTables *d_pf, int n_sm, cudaStream_t stream,
               int *n_launches, const PairProbCommit &pp = PairProbCommit{});
size_t pf_scratch_doubles_per_cta(int W, bool pairprob = false);
// second-generation partition function (pf2.cu): unconstrained windows up to 120 nt, shared-memory resident
bool pf2_supports(const PfLaunch &L);
void pf2_set_enabled(bool on);
size_t pf2_scratch_doubles_per_cta(bool pairprob);
void pf2_upload_tables(const PfTables &q);
void launch_pf2(const PfLaunch &L, const MfeTables *d_mfe, const PfTables *d_pf, int n_sm, cudaStream_t stream,
                int *n_launches, const PairProbCommit &pp);
int pf_grid_size(int W, int n_sm, int n_fold);

constexpr int SHUFFLE_MONO = 0, SHUFFLE_DI = 1;

struct ShuffleLaunch {
    const uint8_t *seq_codes;  // [L] codes of the whole record
    int L, W, step, r, type;
    unsigned long long seed;
    int first_window, n_windows;   // windows of this launch; window w starts at w*step
    int final_slot;                // 1: the last slot is the final-window set (start = L - W), Q5
    long long global_window_base;  // Philox counter base = absolute window index
    uint8_t *out;                  // [(n_windows) * r][W] codes
};
void launch_shuffle(const ShuffleLaunch &L, cudaStream_t stream, int *n_launches);
void launch_gather_windows(const uint8_t *seq_codes, int L, int W, int step, int first_window, int n_windows,
                           int final_slot, uint8_t *out, cudaStream_t stream, int *n_launches);
void launch_slice_hc(const uint8_t *hc, int L, int W, int step, int first_window, int n_windows, int final_slot,
                     uint8_t *out, cudaStream_t stream, int *n_launches);
void launch_slice_sc(const int32_t *es1, int L, int W, int step, int first_window, int n_windows, int final_slot,
                     int32_t *out, cudaStream_t stream, int *n_launches);

// ScanFold-Fold accumulation (accumulate.cu): dense banded accumulators over the nucleotides a shard touches,
// then compaction to per-nucleotide partner lists.
struct AccumDense {
    int nt0, n_nt, W;           // nucleotides [nt0, nt0 + n_nt) (0-based), 2W-1 partner-offset columns each
    int32_t *count;             // [n_nt][2W-1] windows holding the pair
    int32_t *first_seen;        // [n_nt][2W-1] lowest absolute window index (INT32_MAX if none)
    long long *sums;            // [6][n_nt][2W-1]: zA zB mfeA mfeB edA edB (exact split sums, see scanfold_b200.h)
};
struct AccumLaunch {
    int step, first_window, n_windows;
    const int16_t *pair_tbl;    // [n_windows][W]
    const int32_t *z100, *mfe, *ed100;
    AccumDense D;
};
void launch_accumulate(const AccumLaunch &A, cudaStream_t stream, int *n_launches);
// adds `src` (same geometry as rows [row0, row0 + n_rows) of D) into D; first_seen takes the minimum
void launch_accum_merge(const AccumDense &D, int row0, int n_rows, const int32_t *src_count, const int32_t *src_first,
                        const long long *src_sums, cudaStream_t stream, int *n_launches);
// per-nucleotide partner counts for rows [row0, row0 + n_rows) -> nparts[n_rows]; offsets[n_rows + 1] = exclusive scan
void launch_accum_count(const AccumDense &D, int row0, int n_rows, int32_t *nparts, long long *offsets,
                        cudaStream_t stream, int *n_launches);
// exclusive scan of n counts -> offsets[n + 1] (one CTA)
void launch_exclusive_scan(const int32_t *counts, int n, long long *offsets, cudaStream_t stream, int *n_launches);
void launch_accum_emit(const AccumDense &D, int row0, int n_rows, const long long *offsets, int32_t *partner,
                       int32_t *count, int32_t *first_seen, long long *sums, long long n_entries, cudaStream_t stream,
                       int *n_launches);

// Window-averaged base-pair probabilities (pairprob.cu): a dense table over the nucleotides a shard of windows touches,
// W int64 columns per row.  Column 0 of row i sums paired_w(i) = sum_k p^w(i,k) over the windows, column d >= 1 sums
// p^w(i, i+d).  Every term enters as the integer llrint(p * 2^40), so the sums are exact and do not depend on the
// order in which windows, chunks, parts of a scan or GPUs add them.
constexpr double PP_UNIT = 1099511627776.0;   // 2^40
struct PairProbDense {
    int nt0, n_nt, W, step, n_windows;   // rows = nucleotides [nt0, nt0 + n_nt) (0-based); n_windows of the whole record
    long long *cells;                    // [n_nt][W]
};

// The PF kernels' commit of one fold: row i (window coordinates) of the fold's probabilities p(k, l) (k < l) into the
// table rows at `rows` (row i at rows + i * W).  The per-nucleotide sum is formed in a fixed order from the same
// integers that go into the pair columns; the adds are integer reductions.
template <class P>
__device__ __forceinline__ void pp_commit_row(long long *rows, int i, int W, P p) {
    long long *row = rows + (long long)i * W;
    long long paired = 0;
    for (int k = 0; k < i - TURN; k++) paired += llrint(p(k, i) * PP_UNIT);
    for (int l = i + TURN + 1; l < W; l++) {
        const long long v = llrint(p(i, l) * PP_UNIT);
        if (v) atomicAdd(reinterpret_cast<unsigned long long *>(row + (l - i)), (unsigned long long)v);
        paired += v;
    }
    if (paired) atomicAdd(reinterpret_cast<unsigned long long *>(row), (unsigned long long)paired);
}

// rows [row0, row0 + n_rows) of D += src (same layout)
void launch_pairprob_merge(const PairProbDense &D, int row0, int n_rows, const long long *src, cudaStream_t stream,
                           int *n_launches);
// rows [row0, row0 + n_rows): paired[r] = column 0 / n(i); npairs[r] = pairs (i, j) with P(i, j) >= cutoff;
// offsets[n_rows + 1] = their exclusive scan
void launch_pairprob_count(const PairProbDense &D, int row0, int n_rows, double cutoff, double *paired, int32_t *npairs,
                           long long *offsets, cudaStream_t stream, int *n_launches);
// the pairs counted above, row then column order: 1-based i, j and P(i, j)
void launch_pairprob_emit(const PairProbDense &D, int row0, int n_rows, double cutoff, const long long *offsets,
                          int32_t *pi, int32_t *pj, double *prob, cudaStream_t stream, int *n_launches);

}  // namespace sfb
