// Window-averaged base-pair probabilities: reduction and compaction of the table the PF kernels fill (PairProbDense,
// device_common.cuh).  For a scan with window W and step s over a record of n_windows regular windows:
//   P(i,j)    = sum_w p^w(i,j) / n(i,j),   n(i,j) = windows that hold both i and j
//   paired(i) = sum_w sum_k p^w(i,k) / n(i), n(i)   = windows that hold i
// (RNAplfold's averaging with -W W -L W when s = 1).  The window counts are computed here, not stored.  Rows are
// reduced one thread each, in column order, so the pair list comes out sorted by i, then j.
#include "device_common.cuh"

namespace sfb {
namespace {

// regular windows w in [0, n_windows) with w*step <= i and j < w*step + W (i <= j, 0-based)
__device__ __forceinline__ int windows_holding(int i, int j, int W, int step, int n_windows) {
    const int lo = j - W + 1 <= 0 ? 0 : (j - W + 1 + step - 1) / step;
    const int hi = min(i / step, n_windows - 1);
    return hi >= lo ? hi - lo + 1 : 0;
}

__device__ __forceinline__ double average(long long v, int n) { return (double)v * (1.0 / PP_UNIT) / n; }

__global__ void pp_merge_kernel(PairProbDense D, int row0, int n_rows, const long long *src) {
    const long long n = (long long)n_rows * D.W;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n || !src[t]) return;
    D.cells[(long long)row0 * D.W + t] += src[t];
}

__global__ void pp_count_kernel(PairProbDense D, int row0, int n_rows, double cutoff, double *paired, int32_t *npairs) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int W = D.W, i = D.nt0 + row0 + r;
    const long long *row = D.cells + (long long)(row0 + r) * W;
    const int ni = windows_holding(i, i, W, D.step, D.n_windows);
    paired[r] = ni ? average(row[0], ni) : 0.;
    int n = 0;
    for (int d = 1; d < W; d++) {
        const long long v = row[d];
        if (v && average(v, windows_holding(i, i + d, W, D.step, D.n_windows)) >= cutoff) n++;
    }
    npairs[r] = n;
}

__global__ void pp_emit_kernel(PairProbDense D, int row0, int n_rows, double cutoff, const long long *offsets, int32_t *pi,
                               int32_t *pj, double *prob) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int W = D.W, i = D.nt0 + row0 + r;
    const long long *row = D.cells + (long long)(row0 + r) * W;
    long long o = offsets[r];
    for (int d = 1; d < W; d++) {
        const long long v = row[d];
        if (!v) continue;
        const double p = average(v, windows_holding(i, i + d, W, D.step, D.n_windows));
        if (p < cutoff) continue;
        pi[o] = i + 1;
        pj[o] = i + d + 1;
        prob[o] = p;
        o++;
    }
}

}  // namespace

void launch_pairprob_merge(const PairProbDense &D, int row0, int n_rows, const long long *src, cudaStream_t stream,
                           int *n_launches) {
    const long long n = (long long)n_rows * D.W;
    if (n <= 0) return;
    pp_merge_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(D, row0, n_rows, src);
    if (n_launches) (*n_launches)++;
}

void launch_pairprob_count(const PairProbDense &D, int row0, int n_rows, double cutoff, double *paired, int32_t *npairs,
                           long long *offsets, cudaStream_t stream, int *n_launches) {
    if (n_rows <= 0) return;
    pp_count_kernel<<<(n_rows + 127) / 128, 128, 0, stream>>>(D, row0, n_rows, cutoff, paired, npairs);
    if (n_launches) (*n_launches)++;
    launch_exclusive_scan(npairs, n_rows, offsets, stream, n_launches);
}

void launch_pairprob_emit(const PairProbDense &D, int row0, int n_rows, double cutoff, const long long *offsets,
                          int32_t *pi, int32_t *pj, double *prob, cudaStream_t stream, int *n_launches) {
    if (n_rows <= 0) return;
    pp_emit_kernel<<<(n_rows + 127) / 128, 128, 0, stream>>>(D, row0, n_rows, cutoff, offsets, pi, pj, prob);
    if (n_launches) (*n_launches)++;
}

}  // namespace sfb
