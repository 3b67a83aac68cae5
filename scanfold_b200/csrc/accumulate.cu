// ScanFold-Fold accumulation on the device (ScanFold.py:564-677 pair records + :1051-1139 per-partner lists).
//
// Every window contributes one record to each of its W nucleotides: (partner, z, MFE, ED) of that window.
// The reference appends these to Python lists and later sums / averages them per (nucleotide, partner).
// Here one thread owns one nucleotide and walks its <= W/step covering windows in ascending order, adding
// into a banded [n_nt][2W-1] table indexed by partner offset -- a gather, so no atomics and a deterministic
// result.  Values are accumulated EXACTLY: a window value d = k/100 (k integer) enters as the pair
// A = rint(d * 2^20), B = (d - A * 2^-20) * 2^59 (both integers, d == A * 2^-20 + B * 2^-59 exactly), so
// int64 sums of A and B give the exact sum of the doubles the reference adds.  That makes the result
// independent of window order and of how windows are sharded over GPUs (the halo merge is an integer add).
// A second pass compacts the table to per-nucleotide partner lists for the host.
#include <climits>

#include "device_common.cuh"

namespace sfb {
namespace {

__device__ __forceinline__ void split_exact(int k100, long long &a, long long &b) {
    const double d = (double)k100 / 100.0;       // == the double Python's round(x, 2) returns
    const double ra = rint(d * 1048576.0);
    a = (long long)ra;
    b = (long long)((d - ra * (1.0 / 1048576.0)) * 576460752303423488.0);  // 2^59, exact
}

__global__ void accumulate_kernel(AccumLaunch A) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= A.D.n_nt) return;
    const int W = A.D.W, step = A.step, ncol = 2 * W - 1;
    const int k = A.D.nt0 + row;  // 0-based nucleotide
    // windows w (absolute) with w*step <= k < w*step + W, restricted to this shard
    int w_hi = k / step;
    int w_lo = k - W + 1 <= 0 ? 0 : (k - W + 1 + step - 1) / step;
    const int lo = max(w_lo, A.first_window), hi = min(w_hi, A.first_window + A.n_windows - 1);
    const long long plane = (long long)A.D.n_nt * ncol;
    const long long base = (long long)row * ncol;
    for (int w = lo; w <= hi; w++) {
        const int slot = w - A.first_window;
        const int pos = k - w * step;
        const int partner = A.pair_tbl[(long long)slot * W + pos];
        if (partner < 0) continue;   // window without pair records: the all-N short-circuit (Appendix B Q10)
        const int off = partner ? (partner - 1) - pos : 0;
        const long long idx = base + off + (W - 1);
        long long a, b;
        A.D.count[idx] += 1;
        if (w < A.D.first_seen[idx]) A.D.first_seen[idx] = w;
        split_exact(A.z100[slot], a, b);
        A.D.sums[0 * plane + idx] += a;
        A.D.sums[1 * plane + idx] += b;
        split_exact(A.mfe[slot], a, b);
        A.D.sums[2 * plane + idx] += a;
        A.D.sums[3 * plane + idx] += b;
        split_exact(A.ed100[slot], a, b);
        A.D.sums[4 * plane + idx] += a;
        A.D.sums[5 * plane + idx] += b;
    }
}

__global__ void merge_kernel(AccumDense D, int row0, int n_rows, const int32_t *src_count, const int32_t *src_first,
                             const long long *src_sums) {
    const int ncol = 2 * D.W - 1;
    const long long n = (long long)n_rows * ncol;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const long long dst = (long long)row0 * ncol + t;
    const long long plane = (long long)D.n_nt * ncol;
    const int c = src_count[t];
    if (!c) return;
    D.count[dst] += c;
    D.first_seen[dst] = min(D.first_seen[dst], src_first[t]);
    for (int q = 0; q < 6; q++) D.sums[q * plane + dst] += src_sums[q * n + t];
}

__global__ void count_kernel(AccumDense D, int row0, int n_rows, int32_t *nparts) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int ncol = 2 * D.W - 1;
    const int32_t *c = D.count + (long long)(row0 + r) * ncol;
    int n = 0;
    for (int q = 0; q < ncol; q++) n += c[q] != 0;
    nparts[r] = n;
}

// single-CTA exclusive scan (n up to a few million): offsets[0..n]
__global__ void scan_kernel(const int32_t *nparts, int n, long long *offsets) {
    __shared__ long long part[1024];
    const int t = threadIdx.x;
    const int per = (n + 1023) / 1024;
    const int lo = min(n, t * per), hi = min(n, lo + per);
    long long s = 0;
    for (int k = lo; k < hi; k++) s += nparts[k];
    part[t] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        long long v = t >= o ? part[t - o] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    long long run = t ? part[t - 1] : 0;
    for (int k = lo; k < hi; k++) {
        offsets[k] = run;
        run += nparts[k];
    }
    if (t == 1023) offsets[n] = part[1023];
}

__global__ void emit_kernel(AccumDense D, int row0, int n_rows, const long long *offsets, int32_t *partner,
                            int32_t *count, int32_t *first_seen, long long *sums, long long n_entries) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int W = D.W, ncol = 2 * W - 1;
    const long long base = (long long)(row0 + r) * ncol;
    const long long plane = (long long)D.n_nt * ncol;
    long long o = offsets[r];
    const int k1 = D.nt0 + row0 + r + 1;  // 1-based coordinate
    for (int q = 0; q < ncol; q++) {
        const int c = D.count[base + q];
        if (!c) continue;
        partner[o] = k1 + q - (W - 1);
        count[o] = c;
        first_seen[o] = D.first_seen[base + q];
        for (int s = 0; s < 6; s++) sums[s * n_entries + o] = D.sums[s * plane + base + q];
        o++;
    }
}

}  // namespace

void launch_accumulate(const AccumLaunch &A, cudaStream_t stream, int *n_launches) {
    if (A.D.n_nt <= 0 || A.n_windows <= 0) return;
    accumulate_kernel<<<(A.D.n_nt + 127) / 128, 128, 0, stream>>>(A);
    if (n_launches) (*n_launches)++;
}

void launch_accum_merge(const AccumDense &D, int row0, int n_rows, const int32_t *src_count, const int32_t *src_first,
                        const long long *src_sums, cudaStream_t stream, int *n_launches) {
    const long long n = (long long)n_rows * (2 * D.W - 1);
    if (n <= 0) return;
    merge_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(D, row0, n_rows, src_count, src_first, src_sums);
    if (n_launches) (*n_launches)++;
}

void launch_accum_count(const AccumDense &D, int row0, int n_rows, int32_t *nparts, long long *offsets,
                        cudaStream_t stream, int *n_launches) {
    if (n_rows <= 0) return;
    count_kernel<<<(n_rows + 127) / 128, 128, 0, stream>>>(D, row0, n_rows, nparts);
    if (n_launches) (*n_launches)++;
    launch_exclusive_scan(nparts, n_rows, offsets, stream, n_launches);
}

void launch_exclusive_scan(const int32_t *counts, int n, long long *offsets, cudaStream_t stream, int *n_launches) {
    scan_kernel<<<1, 1024, 0, stream>>>(counts, n, offsets);
    if (n_launches) (*n_launches)++;
}

void launch_accum_emit(const AccumDense &D, int row0, int n_rows, const long long *offsets, int32_t *partner,
                       int32_t *count, int32_t *first_seen, long long *sums, long long n_entries, cudaStream_t stream,
                       int *n_launches) {
    if (n_rows <= 0 || n_entries <= 0) return;
    emit_kernel<<<(n_rows + 127) / 128, 128, 0, stream>>>(D, row0, n_rows, offsets, partner, count, first_seen, sums,
                                                         n_entries);
    if (n_launches) (*n_launches)++;
}

}  // namespace sfb
