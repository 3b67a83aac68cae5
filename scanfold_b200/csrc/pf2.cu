// Partition function, second generation: one CTA (512 threads) per window, everything the inner loops touch in
// shared memory, windows up to 120 nt without constraints or with per-nucleotide hard constraints ('x' '<' '>').
//
// Replaces fc.pf(), fc.centroid(), fc.mean_bp_distance() -- ScanFold.py:498,503-504 -- for the native windows of a
// scan; pf.cu keeps enforced pairs, soft constraints and the long windows.
//
// Both passes walk the matrix by COLUMN (3' end): every cell of a column only depends on earlier columns.  r02
// rewrite (the first version spent 6,000 cycles per column in a lane = cell candidate walk whose shared-memory loads
// served one useful lane in three, 3,000 in a serial multiloop sum and three to four barriers per column):
// * separable interior loops: ONE WARP PER PAIRABLE CELL (a compacted list per column), lane = u2, a compile-time
//   loop over u1.  The candidates' weights -- qb (inside) / the outside weight P (outside), already multiplied by the
//   mismatch factor of that pair for the three separable loop classes (generic | 1xn | bulge) -- live in rings
//   [position][column & 31] with a pitch of 33 doubles: the 32 lanes of a load read 32 consecutive doubles (no bank
//   conflict), the u1 step is an immediate offset (no address arithmetic), the size factor K[u1] of lane u2 sits in a
//   register: one LDS.64 + one DFMA per 32 candidates, then one warp reduction per cell.  Lanes 0 and 1 (u2 = 0, 1) read
//   the bulge / 1xn copy, every other lane the generic one; u1 = 0, 1 are peeled the same way.
// * everything else of a column runs beside that walk or in ONE second phase as warp-sized units (two barriers per
//   column): the multiloop sums as row-sliced matrix-vector products with four independent accumulators per lane,
//   the nine table-driven shapes and the hairpin of the NEXT column by item (lane = listed cell, the table loads of an
//   item pair issued together; tabulated tri- / tetra- / hexaloops by a warp-wide key search), the geometric sums as warp
//   scans, the exterior sums, the per-cell outer factors (`prm` rows), the ring bookkeeping; X1 streams PM from L2 two
//   columns ahead on four warps.  Cells are dealt to the warps in weighted rounds by the length of the unit the warp
//   also runs in that phase.  A lone warp in dependent code advances at 10-25 cycles per instruction (LDS 30, a double
//   warp_sum 191, L2 369 cycles: tools/scratch/lat.cu), so the longest per-warp chain of a phase is what is balanced.
// qm lives in a folded triangular matrix with an odd pitch (row and column walks are both bank-conflict free).
// Only qb (read back once per cell) and the multiloop closing weights PM (read as rows) stream through L2.
#include <cstdlib>
#include <type_traits>

#include "device_common.cuh"

namespace sfb {
namespace {

constexpr int P2 = 120;          // longest window
constexpr int PT = 33;           // ring pitch (doubles): [position][column & 31] plus one pad
constexpr int RPAD = 4;          // zero positions either side: a group of four u1 steps may overrun by three
constexpr int RPOS = P2 + 2 * RPAD;
constexpr int RING = RPOS * PT;  // doubles per ring copy
constexpr int PQ = 121;          // pitch of the folded qm matrix (odd)
constexpr int QROWS = (P2 + 3) / 2 + 1;
constexpr int NT2 = 512, NW2 = NT2 / 32;
constexpr int NG = 8;            // inside: partial sums of the multiloop product (one warp each)
constexpr int NH = 5;            // outside: partial sums of H
constexpr int PP = 128;          // pitch of the per-cell arrays
constexpr int PRW = 10;          // doubles per cell parameter row
enum { PR_MMI = 0, PR_MM1, PR_TAU, PR_MLC, PR_FI, PR_F1, PR_FB, PR_FM, PR_ONE, PR_ZERO };

__device__ double g_K2[32 * 32];  // [u2][u1]: size factor of the separable candidate (u1, u2), 0 for the table-driven ones

// the small Boltzmann-factor tables the per-cell code looks up: a shared-memory copy per CTA.  Neighbour codes of the
// stem tables run 0..5, 5 = no neighbour (window border)
struct PfHead {
    double expmismatchI[8][5][5], expmismatch1nI[8][5][5], expmismatch23I[8][5][5], expmismatchH[8][5][5];
    double mlstem[8][6][6];   // E_MLstem factor: mismatchM / dangle5 / dangle3, TerminalAU, MLintern
    double ext[8][6][6];      // exterior stem factor likewise (no MLintern)
    double expstack[8][8];
    double tau[8];            // TerminalAU factor by pair type
    double one, zero, expbulge1, il5;   // il5 = expinternal[5] * expninio[1]  (2x3 loops)
};

struct Smem2 {
    PfHead th;
    double ring[3 * RING];      // generic | 1xn | bulge copies, [position + RPAD][column & 31]
    double ringq[8][P2];        // raw qb (inside) / raw P (outside) of the last columns: table-driven shapes
    double qm[QROWS * PQ + 128]; // folded: row = 3' end k', entries i <= k'-4; the row walks of the matrix-vector units load
                                // up to 65 doubles past the last row's last entry (masked): the pad keeps them inside the array
    double partC[NG][PP];       // partial multiloop sums (inside: qq; outside: H)
    double prm[PP][PRW];        // per listed cell: the outer factors the candidate walk's reduction and stores need
    double partA[PP];           // outside: interior-loop sum of the listed cells
    double partS1a[4][PP];      // table-driven shapes with u2 >= 1 and the hairpin of even columns, by computing warp
    union {
        struct {
            double partS1b[4][PP];   // the same for odd columns
            double partS0[2][PP];    // the two shapes with u2 = 0 (they need the column just finished)
            double qm1[2][PP];
        } in;                        // inside pass only
        double x1buf[2][4][PP];      // outside pass: X1 of a column (partial sums of the four streaming warps), by parity
    } u;
    double ecol[PP];
    double x2[PP], x12[PP], g1[PP];
    double q5[PP], q3[PP];
    double qcol[PP];            // outside: qb of the current column
    double scale[P2 + 40], emlb[PP], ainv[PP];
    double red[32];
    double junk[32];            // store target of the lanes that have nothing to write
    short cen[PP];
    unsigned char S[PP];
    unsigned char Sx[PP + 8];   // Sx[k+1] = code of nucleotide k, Sx[0] = Sx[W+1] = 5
    unsigned char ty[4][PP];    // pair type of the cells of a column (0: not pairable), by column & 3
    unsigned char list[4][PP];  // 5' ends of the cells the candidate walk visits
    unsigned char can5[PP], can3[PP];   // hard constraints: may be the 5' / 3' partner of a pair
    int cnt[4];
#ifdef SFB_PF2_TIMING
    long long tstamp[2][16];
#endif
};
static_assert(sizeof(Smem2) <= 227 * 1024, "one window per SM");

template <int A, int B, class F>
__device__ __forceinline__ void sfor2(F &&f) {
    if constexpr (A <= B) {
        f(std::integral_constant<int, A>{});
        sfor2<A + 1, B>(f);
    }
}

// Separable candidates of one cell: lane = u2, u1 = 0 .. u1max.  pB / p1 / pM point at position u1 = 0 of the bulge /
// 1xn / lane-class copy in this lane's column; inside steps up the positions, outside down.  Returns the lane-class sum
// (u1 >= 2); accB (u1 = 0: bulges) and acc1 (u1 = 1: 1xn loops) take their own outer factor.  From u1 = 15 on only
// lanes 0..15 have candidates (u1 + u2 <= 30): the upper half warp skips the load (one wavefront instead of two).
template <bool OUT>
__device__ __forceinline__ double cand_walk(const double *pB, const double *p1, const double *pM, int u1max, bool lo,
                                            const double (&K)[MAXLOOP + 1], double &accB, double &acc1) {
    constexpr int ST = OUT ? -PT : PT;
    accB = pB[0] * K[0];
    acc1 = p1[ST] * K[1];
    double a0 = 0., a1 = 0.;
    if (u1max >= MAXLOOP) {
        // the full walk (most cells): straight-line code, so the loads run ahead of the DFMAs as far as registers allow
        sfor2<2, MAXLOOP>([&](auto V) {
            constexpr int u1 = decltype(V)::value;
            if (u1 < 15 || lo) {
                if constexpr (u1 & 1)
                    a1 = fma(pM[u1 * ST], K[u1], a1);
                else
                    a0 = fma(pM[u1 * ST], K[u1], a0);
            }
        });
        return a0 + a1;
    }
    sfor2<0, 7>([&](auto Q) {
        constexpr int g = 2 + 4 * decltype(Q)::value;
        if (g <= u1max) {   // warp-uniform
            sfor2<0, 3>([&](auto V) {
                constexpr int u1 = g + decltype(V)::value;
                if constexpr (u1 <= MAXLOOP) {
                    if (u1 < 15 || lo) {
                        if constexpr (u1 & 1)
                            a1 = fma(pM[u1 * ST], K[u1], a1);
                        else
                            a0 = fma(pM[u1 * ST], K[u1], a0);
                    }
                }
            });
        }
    });
    return a0 + a1;
}

__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// the nine shapes as (u1, u2) nibbles: (0,0) (0,1) (1,0) (1,1) (1,2) (2,1) (2,2) (2,3) (3,2)
__host__ __device__ constexpr int shape_u1(int z) { return (int)((0x322211100ull >> (4 * z)) & 15); }
__host__ __device__ constexpr int shape_u2(int z) { return (int)((0x232121010ull >> (4 * z)) & 15); }

// Boltzmann factor of table-driven shape Z (closing pair type t with neighbours si1 = S[i+1], sj1 = S[j-1]; inner pair
// type t2 -- as seen from inside the loop -- with sp1 = S[p-1], sq1 = S[q+1]) without the length scaling (SURVEY A.2)
template <int Z>
__device__ __forceinline__ double shape_f(const PfHead *TH, const PfTables *T, int t, int t2, int si1, int sj1, int sp1, int sq1) {
    constexpr int u1 = shape_u1(Z), u2 = shape_u2(Z);
    constexpr int ul = u1 > u2 ? u1 : u2, us = u1 > u2 ? u2 : u1;
    if constexpr (ul == 0) return TH->expstack[t][t2];
    else if constexpr (us == 0) return TH->expbulge1 * TH->expstack[t][t2];   // bulge of one
    else if constexpr (us == 1 && ul == 1) return T->expint11[t][t2][si1][sj1];
    else if constexpr (us == 1 && u1 == 1) return T->expint21[t][t2][si1][sq1][sj1];
    else if constexpr (us == 1) return T->expint21[t2][t][sq1][si1][sp1];
    else if constexpr (ul == 2) return T->expint22[t][t2][si1][sp1][sq1][sj1];
    else return TH->il5 * TH->expmismatch23I[t][si1][sj1] * TH->expmismatch23I[t2][sq1][sp1];
}

// shape Z closed by (i,j) from inside: weight of the inner pair times the factor; a cell that is no pair has weight 0
template <int Z>
__device__ __forceinline__ double shape_in(const Smem2 &sm, const PfTables *T, int i, int j, int t) {
    constexpr int u1 = shape_u1(Z), u2 = shape_u2(Z);
    const unsigned char *S = sm.S;
    const int p = i + 1 + u1, q = j - 1 - u2;
    const double qpq = sm.ringq[q & 7][p];
    const int t2 = rtype_of(pair_type(S[p], S[q]));
    const double f = shape_f<Z>(&sm.th, T, t, t2, S[i + 1], S[j - 1], S[p - 1], S[q + 1]) * sm.scale[u1 + u2 + 2];
    return qpq != 0. ? qpq * f : 0.;
}

// shape Z around the inner pair (k,l) from outside: (i,j) = (k-1-u1, l+1+u2) is the closing pair
template <int Z>
__device__ __forceinline__ double shape_out(const Smem2 &sm, const PfTables *T, int k, int l, int t2, int W) {
    constexpr int u1 = shape_u1(Z), u2 = shape_u2(Z);
    const unsigned char *S = sm.S;
    const int i = k - 1 - u1, j = l + 1 + u2;
    const bool ok = i >= 0 && j <= W - 1;
    const int ic = max(i, 0), jc = min(j, W - 1);
    const double pij = ok ? sm.ringq[jc & 7][ic] : 0.;
    const int tij = pair_type(S[ic], S[jc]);
    const double f = shape_f<Z>(&sm.th, T, tij, t2, S[ic + 1], S[jc - 1], S[k - 1], S[l + 1]) * sm.scale[u1 + u2 + 2];
    return pij > 0. ? pij * f : 0.;
}

#ifdef SFB_PF2_TIMING
// barrier with bookkeeping: work[slot] += own arrival - release of the previous barrier, wait[slot] += last arrival - own
#define PF2_SYNC(slot)                                                                     \
    {                                                                                      \
        long long now_;                                                                    \
        asm volatile("mov.u64 %0, %%clock64;" : "=l"(now_)::"memory");                     \
        if (lane == 0) sm.tstamp[tpar][warp] = now_;                                       \
        __syncthreads();                                                                   \
        long long m_ = sm.tstamp[tpar][lane & 15];                                         \
        for (int o_ = 8; o_; o_ >>= 1) m_ = max(m_, __shfl_xor_sync(0xffffffffu, m_, o_)); \
        tacc[slot] += now_ - tlast;                                                        \
        tacc[slot + 1] += m_ - now_;                                                       \
        tlast = m_;                                                                        \
        tpar ^= 1;                                                                         \
    }
#define PF2_RESET asm volatile("mov.u64 %0, %%clock64;" : "=l"(tlast)::"memory");
#define PF2_UNIT(k)                                                     \
    {                                                                   \
        long long now_;                                                 \
        asm volatile("mov.u64 %0, %%clock64;" : "=l"(now_)::"memory"); \
        tunit[k] += now_ - tlast;                                       \
    }
#else
#define PF2_UNIT(k)
#define PF2_SYNC(slot) __syncthreads();
#define PF2_RESET
#endif

// PAIRPROB: the launch carries a pair-probability table; the outside pass stages every probability in the CTA's scratch
// (L2 resident) and the fold commits them at its end, when its dG and ED are known to be finite
template <bool PAIRPROB>
__global__ void __launch_bounds__(NT2, 1)
pf2_kernel(PfLaunch L, const MfeTables *__restrict__ MT, const PfTables *__restrict__ T, PairProbCommit pp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem2 &sm = *reinterpret_cast<Smem2 *>(smem_raw);
    const int W = L.W;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const unsigned full = 0xffffffffu;
    double *qbG = L.gscratch + (long long)blockIdx.x * L.gscratch_per_cta;   // qb[j][i], pitch P2
    double *pmG = qbG + P2 * P2;                                              // PM[j][i]
    double *ppG = pmG + P2 * P2;                                              // PAIRPROB: p[l][k]
    const int HF = (W + 3) / 2;
    auto qmrow = [&](int kk) { return kk <= HF ? kk * PQ : (W + 3 - kk) * PQ + (W - kk); };   // + i
#ifdef SFB_PF2_TIMING
    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast;
    int tpar = 0;
    long long tunit[2] = {0, 0};
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(tlast)::"memory");
#endif

    for (int k = tid; k < 200; k += NT2) {
        (&sm.th.expmismatchI[0][0][0])[k] = (&T->expmismatchI[0][0][0])[k];
        (&sm.th.expmismatch1nI[0][0][0])[k] = (&T->expmismatch1nI[0][0][0])[k];
        (&sm.th.expmismatch23I[0][0][0])[k] = (&T->expmismatch23I[0][0][0])[k];
        (&sm.th.expmismatchH[0][0][0])[k] = (&T->expmismatchH[0][0][0])[k];
        if (k < 64) (&sm.th.expstack[0][0])[k] = (&T->expstack[0][0])[k];
        if (k < 8) sm.th.tau[k] = k > 2 ? T->expTermAU : 1.;
    }
    for (int k = tid; k < 8 * 36; k += NT2) {
        const int t = k / 36, a = (k / 6) % 6, b = k % 6;
        double z = 1.;
        double ze = 1.;
        if (a < 5 && b < 5) {
            z = T->expmismatchM[t][a][b];
            ze = T->expmismatchExt[t][a][b];
        } else if (a < 5) {
            z = ze = T->expdangle5[t][a];
        } else if (b < 5) {
            z = ze = T->expdangle3[t][b];
        }
        const double au = t > 2 ? T->expTermAU : 1.;
        sm.th.mlstem[t][a][b] = z * au * T->expMLintern;
        sm.th.ext[t][a][b] = ze * au;
    }
    const PfHead *TH = &sm.th;
    if (tid == 0) {
        sm.th.one = 1.;
        sm.th.zero = 0.;
        sm.th.expbulge1 = T->expbulge[1];
        sm.th.il5 = T->expinternal[5] * T->expninio[1];
        sm.scale[0] = 1.;
        sm.emlb[0] = 1.;
        sm.ainv[0] = 1.;
        const double x = T->expMLbase / T->pf_scale;
        for (int k = 1; k < P2 + 40; k++) sm.scale[k] = sm.scale[k - 1] / T->pf_scale;
        for (int k = 1; k < PP; k++) {
            sm.emlb[k] = sm.emlb[k - 1] * x;
            sm.ainv[k] = sm.ainv[k - 1] / x;
        }
    }
    double K[MAXLOOP + 1];   // size factors of this lane's candidates (lane = u2)
#pragma unroll
    for (int u1 = 0; u1 <= MAXLOOP; u1++) K[u1] = g_K2[lane * 32 + u1];
    __syncthreads();
    const double sc1 = sm.scale[1], sc2 = sm.scale[2], eml1 = sm.emlb[1];
    const double closing = T->expMLclosing;
    const unsigned char *S = sm.S, *Sx = sm.Sx;
    const int cls = lane == 0 ? 2 : (lane == 1 ? 1 : 0);   // ring copy of this lane's candidates with u1 >= 2
    const bool lo = lane < 16;

    // pairable cells of inside column j -> ty / list / cnt of slot j & 3 (one warp)
    auto build_list_inside = [&](int j) {
        const bool c3 = j < W && sm.can3[min(j, PP - 1)];
        const int sj = S[min(j, PP - 1)];
        int t[PP / 32];
#pragma unroll
        for (int b = 0; b < PP / 32; b++) {
            const int i = b * 32 + lane;
            t[b] = (c3 && i <= j - TURN - 1 && sm.can5[i]) ? pair_type(S[i], sj) : 0;
        }
        int n = 0;
#pragma unroll
        for (int b = 0; b < PP / 32; b++) {
            const int i = b * 32 + lane;
            sm.ty[j & 3][i] = (unsigned char)t[b];
            const unsigned m = __ballot_sync(full, t[b] != 0);
            if (t[b]) sm.list[j & 3][n + __popc(m & ((1u << lane) - 1))] = (unsigned char)i;
            n += __popc(m);
        }
        if (lane == 0) sm.cnt[j & 3] = n;
    };
    // outer factors of the listed cells of inside column j (lane = listed cell): what the walk multiplies its class sums
    // with, the multiloop closing factor, the factors of the ring copies / qm1 the cell's qb is stored with
    auto cell_params_inside = [&](int j, int half) {
        if (j >= W) return;
        const int n = sm.cnt[j & 3];
        for (int cc = lane; cc < n; cc += 32) {
            const int i = sm.list[j & 3][cc], t = sm.ty[j & 3][i], t2 = rtype_of(t);
            const int si1 = S[i + 1], sj1 = S[j - 1];
            const bool inner = i > 0 && j < W - 1;   // (i,j) can be the inner pair of an enclosing loop
            const int a = Sx[j + 2] % 5, b = Sx[i] % 5;
            double *r = sm.prm[cc];
            if (half == 0) {
                r[PR_MMI] = TH->expmismatchI[t][si1][sj1];
                r[PR_MM1] = TH->expmismatch1nI[t][si1][sj1];
                r[PR_TAU] = TH->tau[t];
                r[PR_MLC] = closing * TH->mlstem[t2][sj1][si1] * sc2;
                r[PR_ONE] = 1.;
            } else {
                r[PR_FI] = inner ? TH->expmismatchI[t2][a][b] : 0.;
                r[PR_F1] = inner ? TH->expmismatch1nI[t2][a][b] : 0.;
                r[PR_FB] = inner ? TH->tau[t2] : 0.;
                r[PR_FM] = TH->mlstem[t][Sx[i]][Sx[j + 2]];
                r[PR_ZERO] = 0.;
            }
        }
    };
    // hairpin closed by (i,j) (SURVEY A.2): the general formula per lane; loops of 3, 4 and 6 nucleotides are left to
    // special_hairpins (tabulated tri- / tetra- / hexaloops)
    auto hairpin_f = [&](int i, int j, int t) {
        const int u = j - i - 1;
        if (u == 3 || u == 4 || u == 6) return 0.;
        return T->exphairpin_len[u] * TH->expmismatchH[t][S[i + 1]][S[j - 1]];
    };
    // the three cells of column j that close a loop of 3, 4 or 6: the key tables are searched by the whole warp (first
    // match in table order wins, as in the serial search); adds the hairpin term to the cell's slice
    auto special_hairpins = [&](int j, double(*ps)[PP]) {
        double val[3];
        bool have[3];
#pragma unroll
        for (int z = 0; z < 3; z++) {
            const int u = z == 0 ? 3 : (z == 1 ? 4 : 6), i = j - u - 1;
            const int t = i >= 0 ? sm.ty[j & 3][i] : 0;
            have[z] = t != 0;
            val[z] = 0.;
            if (have[z]) {   // warp-uniform
                const int key = loop_key_dev(S, i, u + 2);
                const int n = z == 0 ? MT->n_tri : (z == 1 ? MT->n_tetra : MT->n_hexa);
                const int *keys = z == 0 ? MT->tri_key : (z == 1 ? MT->tetra_key : MT->hexa_key);
                const unsigned m0 = __ballot_sync(full, lane < n && keys[lane] == key);
                const unsigned m1 = __ballot_sync(full, lane + 32 < n && keys[lane + 32] == key);
                const int hit = m0 ? __ffs(m0) - 1 : (m1 ? 32 + __ffs(m1) - 1 : -1);
                const double z0 = T->exphairpin_len[u];
                if (hit >= 0)
                    val[z] = z == 0 ? T->exptri[hit] : (z == 1 ? T->exptetra[hit] : T->exphexa[hit]);
                else
                    val[z] = z == 0 ? z0 * TH->tau[t] : z0 * TH->expmismatchH[t][S[i + 1]][S[j - 1]];
            }
        }
        __syncwarp();
#pragma unroll
        for (int z = 0; z < 3; z++) {
            const int u = z == 0 ? 3 : (z == 1 ? 4 : 6), i = j - u - 1;
            if (have[z] && lane == 0) ps[3][i] += val[z] * sm.scale[u + 2];
        }
    };
    // shapes with u2 >= 1 and the hairpin of inside column j: w = 0..2 two shapes each, 3 the hairpin, 4 the 1x1 loops;
    // lane = listed cell
    auto shapes1_unit = [&](int j, int w) {
        if (j >= W) return;
        const int n = sm.cnt[j & 3];
        for (int cc = lane; cc < n; cc += 32) {
            const int i = sm.list[j & 3][cc], t = sm.ty[j & 3][i];
            double v;
            if (w == 0)
                v = shape_in<6>(sm, T, i, j, t) + shape_in<1>(sm, T, i, j, t);
            else if (w == 1)
                v = shape_in<4>(sm, T, i, j, t) + shape_in<7>(sm, T, i, j, t);
            else if (w == 2)
                v = shape_in<5>(sm, T, i, j, t) + shape_in<8>(sm, T, i, j, t);
            else if (w == 3)
                v = hairpin_f(i, j, t) * sm.scale[j - i + 1];
            else
                v = shape_in<3>(sm, T, i, j, t);
            if (w < 4)
                (j & 1 ? sm.u.in.partS1b : sm.partS1a)[w][i] = v;
            else
                (j & 1 ? sm.g1 : sm.x12)[i] = v;   // fifth slice: two arrays only the outside pass uses
        }
        if (w == 3) {
            __syncwarp();
            special_hairpins(j, j & 1 ? sm.u.in.partS1b : sm.partS1a);
        }
    };
    // the two shapes with u2 = 0 (stack, bulge of one on the 5' side) of inside column j, w = 0 / 1
    auto shapes0_unit = [&](int j, int w) {
        if (j >= W) return;
        const int n = sm.cnt[j & 3];
        for (int cc = lane; cc < n; cc += 32) {
            const int i = sm.list[j & 3][cc], t = sm.ty[j & 3][i];
            sm.u.in.partS0[w][i] = w == 0 ? shape_in<0>(sm, T, i, j, t) : shape_in<2>(sm, T, i, j, t);
        }
    };

    for (int fold = blockIdx.x; fold < L.n_fold; fold += gridDim.x) {
        __syncthreads();
        for (int k = tid; k < PP; k += NT2) {
            const bool in = k < W;
            const int code = in ? L.seqs[(long long)fold * W + k] : 4;
            sm.S[k] = (unsigned char)code;
            if (k + 1 < PP + 8) sm.Sx[k + 1] = (unsigned char)(in ? code : 5);
            if (k == 0) sm.Sx[0] = 5;
            const char ch = (L.hc && in) ? (char)L.hc[(long long)fold * W + k] : '.';
            sm.can5[k] = in && !(ch == 'x' || ch == '>');
            sm.can3[k] = in && !(ch == 'x' || ch == '<');
            sm.cen[k] = 0;
            sm.u.in.qm1[0][k] = 0.;
            sm.u.in.qm1[1][k] = 0.;
            sm.ecol[k] = 0.;
            sm.x2[k] = 0.;
            sm.x12[k] = 0.;
            sm.g1[k] = 0.;
            sm.partA[k] = 0.;
            sm.u.in.partS0[0][k] = 0.;
            sm.u.in.partS0[1][k] = 0.;
        }
        for (int k = tid; k < 3 * RING; k += NT2) sm.ring[k] = 0.;
        for (int k = tid; k < 8 * P2; k += NT2) (&sm.ringq[0][0])[k] = 0.;
        for (int k = tid; k < NG * PP; k += NT2) (&sm.partC[0][0])[k] = 0.;
        for (int k = tid; k < 4 * PP; k += NT2) {
            (&sm.partS1a[0][0])[k] = 0.;
            (&sm.u.in.partS1b[0][0])[k] = 0.;
        }
        if (tid == 0) {
            sm.q5[0] = 1.;
            for (int k = 1; k <= min(W, TURN + 1); k++) sm.q5[k] = sm.q5[k - 1] * sc1;
        }
        __syncthreads();
        if (warp == 14) build_list_inside(TURN + 1);
        if (warp == 15) build_list_inside(TURN + 2);
        __syncthreads();
        if (warp >= 8 && warp < 13) shapes1_unit(TURN + 1, warp - 8);   // hairpins: all the first column can close
        if (warp == 14 || warp == 15) cell_params_inside(TURN + 1, warp - 14);
        __syncthreads();
        PF2_RESET
        // ================= inside, column j =================
        for (int j = TURN + 1; j < W; j++) {
            const int par = j & 1, sl = j & 3;
            // ---- phase 1: the candidate walk of the pairable cells (all warps); first, beside it: shapes with u2 >= 1
            // of the next column (warps 8-11), the cells that are no pair and qm of the previous column (warps 12-15)
            if (warp >= 12) {
                const int i = tid - 12 * 32;
                if (!sm.ty[sl][i] && i < P2) {
                    sm.ringq[j & 7][i] = 0.;
                    if (i < W) qbG[j * P2 + i] = 0.;
                    sm.u.in.qm1[par][i] = i <= j - TURN - 2 ? sm.u.in.qm1[par ^ 1][i] * eml1 : 0.;
                }
                if (j - 1 > TURN && i <= j - TURN - 2) {
                    double qq = 0.;
#pragma unroll
                    for (int g = 0; g < NG; g++) qq += sm.partC[g][i];
                    sm.qm[qmrow(j - 1) + i] = sm.u.in.qm1[par ^ 1][i] + sm.ecol[i] + qq;
                }
                if (warp == 15) build_list_inside(j + 2);
                if (warp == 12) shapes1_unit(j + 1, 4);
            } else if (warp >= 8) {
                shapes1_unit(j + 1, warp - 8);
            }
            PF2_UNIT(0)
            {
                const int n = sm.cnt[sl];
                const double *qm1p = sm.u.in.qm1[par ^ 1];
                // per-lane roles (no divergence inside the cell loop): what the lane adds to the reduction beside its
                // candidates -- lanes 0..NG-1 a partial sum of the multiloop closed by (i,j) (previous column's products),
                // the next seven a slice of the table-driven shapes -- and what it stores once qb is known: ring copies
                // (lanes 0-2), the raw copy (3), qm1 (4)
                const double *ebase = lane < NG ? &sm.partC[lane][1]
                                                : (lane < NG + 4 ? &(par ? sm.u.in.partS1b : sm.partS1a)[lane - NG][0]
                                                                 : (lane == NG + 4 ? (par ? sm.g1 : sm.x12)
                                                                                   : (lane < NG + 7 ? &sm.u.in.partS0[lane - NG - 5][0] : &sm.prm[0][PR_ZERO])));
                const int estride = lane < NG + 7 ? 1 : 0;
                const int ixE = lane < NG ? PR_MLC : PR_ONE;
                const int ixM = lane == 0 ? PR_TAU : (lane == 1 ? PR_MM1 : PR_MMI);
                const int ixF = lane < 3 ? PR_FI + lane : (lane == 3 ? PR_ONE : (lane == 4 ? PR_FM : PR_ZERO));
                double *dbase = lane < 3 ? &sm.ring[lane * RING + RPAD * PT + (j & 31)]
                                         : (lane == 3 ? &sm.ringq[j & 7][0] : (lane == 4 ? &sm.u.in.qm1[par][0] : &sm.junk[lane]));
                const int dstride = lane < 3 ? PT : (lane < 5 ? 1 : 0);
                const double emlL = lane == 4 ? eml1 : 0.;
                // the cells are dealt in rounds of 26, by what else the warp does in this phase: warps 0-7 (no unit) and 13-14
                // (the short one) take two, the shape warps 8-12 and the list builder 15 one
                const int o1 = warp < 8 ? warp : (warp < 13 ? warp + 12 : (warp < 15 ? warp - 5 : 25));
                const int o2 = warp < 8 ? warp + 10 : ((warp == 13 || warp == 14) ? warp + 5 : 1 << 20);
                for (int c0 = o1; c0 < n; c0 = (c0 % 26 == o1 && o2 < 26) ? c0 - o1 + o2 : c0 - c0 % 26 + 26 + o1) {
                    const int cc = c0;
                    const int i = sm.list[sl][cc];
                    const double *r = sm.prm[cc];
                    const double tau = r[PR_TAU], mm1 = r[PR_MM1];
                    const double mulM = r[ixM], ext = ebase[i * estride] * r[ixE], fm = r[ixF];
                    const double fa = i <= j - TURN - 2 ? qm1p[i] * emlL : 0.;
                    const double *pb = sm.ring + (i + 1 + RPAD) * PT + ((j - 1 - min(lane, MAXLOOP)) & 31);   // (lane 31 has no candidate: not the column being written)
                    double accB, acc1;
                    const double aM = cand_walk<false>(pb + 2 * RING, pb + RING, pb + cls * RING, min(MAXLOOP, j - i - 6), lo, K, accB, acc1);
                    double v = aM * mulM + accB * tau + acc1 * mm1 + ext;
                    v = warp_sum(v);
                    dbase[i * dstride] = fma(v, fm, fa);
                    if (lane == 3) qbG[j * P2 + i] = v;
                }
            }
            PF2_SYNC(0)
            // ---- phase 2: one unit per warp
            const double *qm1c = sm.u.in.qm1[par];
            if (warp < NG) {
                // qq[i] = sum_k' qm[i,k'-1] qm1[k',j]: rows k' = 4 + warp, + NG, ..; lane = cell in four blocks
                double a0 = 0., a1 = 0., a2 = 0., a3 = 0.;
#pragma unroll 4
                for (int kk = 4 + warp; kk <= j - 5; kk += NG) {
                    const double w = qm1c[kk + 1];
                    const double *row = sm.qm + qmrow(kk) + lane;
                    const int lim = kk - 4 - lane;   // cell i = 32 b + lane takes part if 32 b <= lim
                    const double v0 = row[0], v1 = row[32], v2 = row[64], v3 = row[96];
                    a0 = fma(lim >= 0 ? v0 : 0., w, a0);
                    a1 = fma(lim >= 32 ? v1 : 0., w, a1);
                    a2 = fma(lim >= 64 ? v2 : 0., w, a2);
                    a3 = fma(lim >= 96 ? v3 : 0., w, a3);
                }
                sm.partC[warp][lane] = a0;
                sm.partC[warp][lane + 32] = a1;
                sm.partC[warp][lane + 64] = a2;
                sm.partC[warp][lane + 96] = a3;
            } else if (warp < NG + 2) {
                shapes0_unit(j + 1, warp - NG);
            } else if (warp == 10) {
                // E[i] = sum_{k=i+1}^{j-4} eMLb[k-i] qm1[k,j] = ainv[i] * (suffix sum of eMLb[k] qm1[k,j])
                double tk[4], tot = 0.;
#pragma unroll
                for (int z = 0; z < 4; z++) {
                    const int k = 4 * lane + z;
                    tk[z] = (k <= j - TURN - 1 && k < P2) ? sm.emlb[k] * qm1c[k] : 0.;
                    tot += tk[z];
                }
                double inc = tot;
                for (int o = 1; o < 32; o <<= 1) {
                    const double u = __shfl_down_sync(full, inc, o);
                    if (lane + o < 32) inc += u;
                }
                double run = __shfl_down_sync(full, inc, 1);
                if (lane == 31) run = 0.;
#pragma unroll
                for (int z = 3; z >= 0; z--) {
                    const int k = 4 * lane + z;
                    if (k < P2) sm.ecol[k] = run * sm.ainv[k];
                    run += tk[z];
                }
            } else if (warp == 11) {
                double acc = 0.;
                const int n = sm.cnt[sl];
                for (int cc = lane; cc < n; cc += 32) {
                    const int i = sm.list[sl][cc];
                    acc += sm.q5[i] * sm.ringq[j & 7][i] * TH->ext[sm.ty[sl][i]][Sx[i]][Sx[j + 2]];
                }
                acc = warp_sum(acc);
                if (lane == 0) sm.q5[j + 1] = sm.q5[j] * sc1 + acc;
            } else if (warp == 12) {
                // the ring column the next column writes: its last reader (column j) is done
                const int slot = (j + 1) & 31;
                for (int p = lane; p < RPOS; p += 32) {
                    sm.ring[p * PT + slot] = 0.;
                    sm.ring[RING + p * PT + slot] = 0.;
                    sm.ring[2 * RING + p * PT + slot] = 0.;
                }
            } else if (warp == 13 || warp == 14) {
                cell_params_inside(j + 1, warp - 13);
            }
            PF2_SYNC(2)
        }
        const double Z = sm.q5[W], invZ = 1. / Z;

        // ================= outside, column l =================
        for (int k = tid; k < 3 * RING; k += NT2) sm.ring[k] = 0.;
        for (int k = tid; k < 8 * P2; k += NT2) (&sm.ringq[0][0])[k] = 0.;
        for (int k = tid; k < NG * PP; k += NT2) (&sm.partC[0][0])[k] = 0.;
        for (int k = tid; k < 4 * PP; k += NT2) (&sm.partS1a[0][0])[k] = 0.;
        for (int k = tid; k < 2 * 4 * PP; k += NT2) (&sm.u.x1buf[0][0][0])[k] = 0.;
        if (tid < PP) sm.x12[tid] = sm.ecol[tid] = 0.;   // x12: the inside pass used it as a shape slice; ecol: fifth slice here
        if (tid < PP) sm.qcol[tid] = (tid <= W - 1 - TURN - 1) ? qbG[(W - 1) * P2 + tid] : 0.;   // qb of the first outside column
        if (tid == 0) {
            sm.q3[W] = 1.;
            for (int k = W - 1; k >= max(0, W - TURN - 1); k--) sm.q3[k] = sm.q3[k + 1] * sc1;
            sm.cnt[(W - 1) & 3] = 0;   // cells of the last column have no enclosing pair
        }
        double ed_local = 0.;
        __syncthreads();
        PF2_RESET
        for (int l = W - 1; l > TURN; l--) {
            const int sl = l & 3;
            // X1[i,l-2] = sum_{j >= l+4} PM[i,j] qm[l-1,j-1] two columns ahead (PM of those columns is final): warps 12-15
            // take the rows j = l+4+w, +4, .. of all cells (lane = cell in up to four blocks), streamed from L2 with two
            // rows (up to eight loads) in flight; most rows before the barrier, the rest after it; partial sums per warp
            const int lx = l - 2, xw = warp - 12;
            const int xj0 = lx + 6, xjm = W;   // (all rows before the barrier: that phase is the longer one)
            double xa[4] = {0., 0., 0., 0.};
            auto x1_rows = [&](int ja, int jb) {
                if (lx <= TURN) return;
                const int imax = lx - TURN - 1;
                const int nb4 = imax / 32 + 1;   // blocks of cells that exist
                const double *pr = pmG + lane;
                const double *qv = sm.qm + lx + 1;
                int j = ja + xw;
                for (; j + 4 < jb; j += 8) {
                    double pv[8];
#pragma unroll
                    for (int z = 0; z < 4; z++) {
                        pv[z] = z < nb4 ? pr[j * P2 + 32 * z] : 0.;
                        pv[4 + z] = z < nb4 ? pr[(j + 4) * P2 + 32 * z] : 0.;
                    }
                    const double w0 = qv[qmrow(j - 1)], w1 = qv[qmrow(j + 3)];
#pragma unroll
                    for (int z = 0; z < 4; z++) xa[z] = fma(pv[4 + z], w1, fma(pv[z], w0, xa[z]));
                }
                for (; j < jb; j += 4) {
                    const double w0 = qv[qmrow(j - 1)];
#pragma unroll
                    for (int z = 0; z < 4; z++) xa[z] = fma(z < nb4 ? pr[j * P2 + 32 * z] : 0., w0, xa[z]);
                }
            };
            // ---- phase 1: one unit per warp, then (warps 0-11) the candidate walk of the listed cells
            if (warp < 5) {
                // table-driven shapes closed outside (k,l), two per warp (the last one), lane = listed cell
                const int n = sm.cnt[sl];
                for (int cc = lane; cc < n; cc += 32) {
                    const int k = sm.list[sl][cc];
                    const int t2 = rtype_of(pair_type(S[k], S[l]));
                    double v;
                    if (warp == 0)
                        v = shape_out<6>(sm, T, k, l, t2, W) + shape_out<1>(sm, T, k, l, t2, W);
                    else if (warp == 1)
                        v = shape_out<4>(sm, T, k, l, t2, W) + shape_out<7>(sm, T, k, l, t2, W);
                    else if (warp == 2)
                        v = shape_out<5>(sm, T, k, l, t2, W) + shape_out<8>(sm, T, k, l, t2, W);
                    else if (warp == 3)
                        v = shape_out<3>(sm, T, k, l, t2, W) + shape_out<0>(sm, T, k, l, t2, W);
                    else
                        v = shape_out<2>(sm, T, k, l, t2, W);
                    (warp < 4 ? sm.partS1a[warp] : sm.ecol)[k] = v;
                }
            } else if (warp == 5) {
                // G1[k] = sum_{i<k} X1[i] eMLb[k-1-i] = eMLb[k-1] * (prefix sum of X1[i] ainv[i])
                const double(*x1c)[PP] = sm.u.x1buf[l & 1];
                double tk[4], tot = 0.;
#pragma unroll
                for (int z = 0; z < 4; z++) {
                    const int i = 4 * lane + z;
                    tk[z] = (i <= l - TURN - 1 && i < P2) ? (x1c[0][i] + x1c[1][i] + x1c[2][i] + x1c[3][i]) * sm.ainv[i] : 0.;
                    tot += tk[z];
                }
                double inc = tot;
                for (int o = 1; o < 32; o <<= 1) {
                    const double u = __shfl_up_sync(full, inc, o);
                    if (lane >= o) inc += u;
                }
                double run = __shfl_up_sync(full, inc, 1);
                if (lane == 0) run = 0.;
#pragma unroll
                for (int z = 0; z < 4; z++) {
                    const int k = 4 * lane + z;
                    if (k < P2) sm.g1[k] = k >= 1 ? run * sm.emlb[k - 1] : 0.;
                    run += tk[z];
                }
            } else if (warp == 6) {
                // q3[l] for the next column
                double a3 = 0.;
                for (int j = l + TURN + 1 + lane; j < W; j += 32) {
                    const double q = qbG[j * P2 + l];
                    a3 += q * sm.q3[j + 1] * TH->ext[pair_type(S[l], S[j])][Sx[l]][Sx[j + 2]];
                }
                a3 = warp_sum(a3);
                if (lane == 0) sm.q3[l] = sm.q3[l + 1] * sc1 + a3;
            } else if (warp < 7 + NH) {
                // H[k] = sum_{i <= k-6} (X1+X2)[i] qm[i+1,k-1]: i = g, g + NH, ..; lane = cell in four blocks
                const int g = warp - 7;
                double a0 = 0., a1 = 0., a2 = 0., a3 = 0.;
                const int kmax = l - TURN - 1;   // cells k <= kmax
                const double *r0 = sm.qm + qmrow(max(lane - 1, 0)) + 1, *r1 = sm.qm + qmrow(lane + 31) + 1;
                const double *r2 = sm.qm + qmrow(min(lane + 63, W - 1)) + 1, *r3 = sm.qm + qmrow(min(lane + 95, W - 1)) + 1;
                const int l0 = min(lane, kmax + 0 >= lane ? lane : -100) - 6;   // cell k = lane + 32 b: terms i <= k - 6
                const int m0 = lane <= kmax ? lane - 6 : -1, m1 = lane + 32 <= kmax ? lane + 26 : -1;
                const int m2 = lane + 64 <= kmax ? lane + 58 : -1, m3 = lane + 96 <= kmax ? lane + 90 : -1;
                (void)l0;
#pragma unroll 4
                for (int i = g; i <= l - 10; i += NH) {
                    const double w = sm.x12[i];
                    const double v0 = r0[i], v1 = r1[i], v2 = r2[i], v3 = r3[i];
                    a0 = fma(i <= m0 ? v0 : 0., w, a0);
                    a1 = fma(i <= m1 ? v1 : 0., w, a1);
                    a2 = fma(i <= m2 ? v2 : 0., w, a2);
                    a3 = fma(i <= m3 ? v3 : 0., w, a3);
                }
                sm.partC[g][lane] = a0;
                sm.partC[g][lane + 32] = a1;
                sm.partC[g][lane + 64] = a2;
                sm.partC[g][lane + 96] = a3;
            } else {
                x1_rows(xj0, xjm);
            }
            PF2_UNIT(1)
            {
                const int n = sm.cnt[sl];
                const int ixM = lane == 0 ? PR_TAU : (lane == 1 ? PR_MM1 : PR_MMI);
                // the cells are dealt in rounds of 23 by the length of the warp's unit, shortest first (4 5 6 8 9 10 11 | 7 0 1 2 3
                // | X1 streamers 12-15); the first seven take a second one
                const int o1 = warp == 4 ? 0 : (warp == 5 ? 1 : (warp == 6 ? 2 : (warp >= 8 && warp < 12 ? warp - 5 : (warp == 7 ? 7 : (warp < 4 ? warp + 8 : warp)))));
                const int o2 = o1 < 7 ? o1 + 16 : 1 << 20;
                for (int cc = o1; cc < n; cc = (cc % 23 == o1 && o2 < 23) ? cc - o1 + o2 : cc - cc % 23 + 23 + o1) {
                    const int k = sm.list[sl][cc];
                    const int t2 = rtype_of(pair_type(S[k], S[l])), a = S[l + 1], b = S[k - 1];
                    const double mmI = TH->expmismatchI[t2][a][b], mm1 = TH->expmismatch1nI[t2][a][b], tau = TH->tau[t2];
                    const double mulM = ixM == PR_TAU ? tau : (ixM == PR_MM1 ? mm1 : mmI);
                    const double *pb = sm.ring + (k - 1 + RPAD) * PT + ((l + 1 + min(lane, MAXLOOP)) & 31);
                    double accB, acc1;
                    const double aM = cand_walk<true>(pb + 2 * RING, pb + RING, pb + cls * RING, min(MAXLOOP, k - 1), lo, K, accB, acc1);
                    double v = aM * mulM + accB * tau + acc1 * mm1;
                    v = warp_sum(v);
                    if (lane == 0) sm.partA[k] = v;
                }
            }
            PF2_SYNC(4)
            // ---- phase 2: P of the column, ring copies, PM, probabilities; X2 and qb of the next column
            if (tid < PP) {
                const int k = tid;
                double Pv = 0., vG = 0., v1 = 0., vB = 0., pm = 0., pk = 0.;
                if (k <= l - TURN - 1) {
                    const double qkl = sm.qcol[k];
                    if (qkl != 0.) {
                        const int t = pair_type(S[k], S[l]);
                        const double fx = TH->ext[t][Sx[k]][Sx[l + 2]];
                        if (k >= 1 && l <= W - 2) {
                            Pv = sm.partA[k] + sm.partS1a[0][k] + sm.partS1a[1][k] + sm.partS1a[2][k] + sm.partS1a[3][k] + sm.ecol[k];
                            double ml = sm.g1[k];
#pragma unroll
                            for (int g = 0; g < NH; g++) ml += sm.partC[g][k];
                            Pv += ml * TH->mlstem[t][Sx[k]][Sx[l + 2]] * sc2;
                        }
                        Pv += sm.q5[k] * sm.q3[l + 1] * invZ * fx;
                        if (Pv != 0.) {
                            const int a = S[k + 1], b = S[l - 1];
                            vG = Pv * TH->expmismatchI[t][a][b];
                            v1 = Pv * TH->expmismatch1nI[t][a][b];
                            vB = Pv * TH->tau[t];
                        }
                        pm = Pv * closing * TH->mlstem[rtype_of(t)][S[l - 1]][S[k + 1]];
                        const double p = Pv * qkl;
                        pk = p;
                        ed_local += p * (1. - p);
                        if (p > 0.5) {
                            sm.cen[k] = (short)(l + 1);
                            sm.cen[l] = (short)(k + 1);
                        }
                        if (L.bpp) L.bpp[((long long)fold * W + k) * W + l] = p;
                    }
                    pmG[l * P2 + k] = pm;
                    if constexpr (PAIRPROB) ppG[l * P2 + k] = pk;
                }
                if (k < P2) {
                    const int o = (k + RPAD) * PT + (l & 31);
                    sm.ring[o] = vG;
                    sm.ring[RING + o] = v1;
                    sm.ring[2 * RING + o] = vB;
                    sm.ringq[l & 7][k] = Pv;
                }
                // the next column l-1: X1 (streamed two columns ago), X2 by its recurrence, qb
                const int ln = l - 1;
                double x1 = 0., x2 = 0., qn = 0.;
                if (ln > TURN && k <= ln - TURN - 1) {
                    x1 = sm.u.x1buf[ln & 1][0][k] + sm.u.x1buf[ln & 1][1][k] + sm.u.x1buf[ln & 1][2][k] + sm.u.x1buf[ln & 1][3][k];
                    x2 = sm.x2[k] * eml1 + pm;
                    qn = qbG[ln * P2 + k];
                }
                sm.x2[k] = x2;
                sm.x12[k] = x1 + x2;
                sm.qcol[k] = qn;
            } else if (warp == 4) {
                // cells of the next column the candidate walk visits (qb != 0, an enclosing pair exists) and their outer
                // factors
                const int ln = l - 1;
                double q[PP / 32];
#pragma unroll
                for (int b = 0; b < PP / 32; b++) {
                    const int k = b * 32 + lane;
                    q[b] = (ln > TURN && k >= 1 && k <= ln - TURN - 1) ? qbG[ln * P2 + k] : 0.;
                }
                int n = 0;
#pragma unroll
                for (int b = 0; b < PP / 32; b++) {
                    const bool on = q[b] != 0.;
                    const unsigned m = __ballot_sync(full, on);
                    if (on) sm.list[ln & 3][n + __popc(m & ((1u << lane) - 1))] = (unsigned char)(b * 32 + lane);
                    n += __popc(m);
                }
                if (lane == 0) sm.cnt[ln & 3] = n;
            } else if (warp >= 12) {
                x1_rows(xjm, W);
                const int imax = lx - TURN - 1;   // cells beyond the column's last one read stale PM: dropped here
#pragma unroll
                for (int z = 0; z < 4; z++) sm.u.x1buf[lx & 1][xw][32 * z + lane] = (lx > TURN && 32 * z + lane <= imax) ? xa[z] : 0.;
            }
            PF2_SYNC(6)
        }

        // ================= ED, centroid =================
        ed_local = warp_sum(ed_local);
        if (lane == 0) sm.red[warp] = ed_local;
        __syncthreads();
        if (tid == 0) {
            double s = 0.;
            for (int w = 0; w < NW2; w++) s += sm.red[w];
            const double dG = (-log(Z) - W * log(T->pf_scale)) * T->kT / 1000.;
            L.ed[fold] = 2. * s;
            L.dG[fold] = dG;
            if (L.n_out_of_range && !(isfinite(dG) && isfinite(2. * s))) atomicAdd(L.n_out_of_range, 1);
        }
        for (int k = tid; k < W; k += NT2) L.centroid[(long long)fold * W + k] = sm.cen[k];
        if constexpr (PAIRPROB) {
            // every thread forms the sum and dG as thread 0 did: commit only what the fold's outputs say is in range
            double s = 0.;
            for (int w = 0; w < NW2; w++) s += sm.red[w];
            const double dG = (-log(Z) - W * log(T->pf_scale)) * T->kT / 1000.;
            if (isfinite(dG) && isfinite(2. * s) && tid < W)
                pp_commit_row(pp.table + (pp.row0 + (long long)fold * pp.step) * W, tid, W,
                              [&](int k, int l) { return ppG[l * P2 + k]; });
        }
#ifdef SFB_PF2_TIMING
        if (blockIdx.x == 0 && fold == 0 && lane == 0)
            printf("pf2 timing warp %2d: inside p1 %lld wait %lld p2 %lld wait %lld | outside p1 %lld wait %lld p2 %lld wait %lld\n", warp,
                   tacc[0], tacc[1], tacc[2], tacc[3], tacc[4], tacc[5], tacc[6], tacc[7]);
        if (blockIdx.x == 0 && fold == 0 && lane == 0)
            printf("pf2 units  warp %2d: inside p1 unit %lld | outside p1 unit %lld\n", warp, tunit[0], tunit[1]);
#endif
    }
}

}  // namespace

static bool &pf2_enabled() {
    static bool on = !(getenv("SFB_PF_ENGINE") && atoi(getenv("SFB_PF_ENGINE")) == 1);
    return on;
}
void pf2_set_enabled(bool on) { pf2_enabled() = on; }

bool pf2_supports(const PfLaunch &L) {
    return pf2_enabled() && (!L.hc || L.hc_simple) && !L.sc && L.max_span <= 0 && L.pf_scale <= 0. && L.W >= 2 * TURN + 4 &&
           L.W <= P2;   // the scale is baked into g_K2 and the shared scale row: a rescaled retry runs on pf.cu
}

size_t pf2_scratch_doubles_per_cta(bool pairprob) { return (pairprob ? 3 : 2) * (size_t)P2 * P2; }

void pf2_upload_tables(const PfTables &q) {
    static double kk[32 * 32];
    double scale[40];
    scale[0] = 1.;
    for (int k = 1; k < 40; k++) scale[k] = scale[k - 1] / q.pf_scale;
    for (int u2 = 0; u2 < 32; u2++)
        for (int u1 = 0; u1 < 32; u1++) {
            const int u = u1 + u2, us = u1 < u2 ? u1 : u2, ul = u1 < u2 ? u2 : u1;
            double v = 0.;
            if (u <= MAXLOOP) {
                if (us == 0) {
                    if (ul >= 2) v = q.expbulge[ul] * scale[u + 2];                                 // bulge
                } else if (us == 1) {
                    if (ul >= 3) v = q.expinternal[u] * q.expninio[ul - 1] * scale[u + 2];           // 1xn
                } else if (!(us == 2 && ul <= 3)) {
                    v = q.expinternal[u] * q.expninio[ul - us] * scale[u + 2];                       // generic
                }
            }
            kk[u2 * 32 + u1] = v;
        }
    cudaMemcpyToSymbol(g_K2, kk, sizeof(kk));
}

void launch_pf2(const PfLaunch &L, const MfeTables *d_mfe, const PfTables *d_pf, int n_sm, cudaStream_t stream,
                int *n_launches, const PairProbCommit &pp) {
    const size_t smem = sizeof(Smem2);
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(pf2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(pf2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        configured = true;
    }
    const int grid = L.n_fold < n_sm ? L.n_fold : n_sm;
    if (pp.table)
        pf2_kernel<true><<<grid, NT2, smem, stream>>>(L, d_mfe, d_pf, pp);
    else
        pf2_kernel<false><<<grid, NT2, smem, stream>>>(L, d_mfe, d_pf, pp);
    if (n_launches) (*n_launches)++;
}

}  // namespace sfb
