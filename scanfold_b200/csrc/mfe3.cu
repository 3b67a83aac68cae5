// MFE fold kernel, third generation: one CTA per fold, int16 energies, windows up to 300 nt; energy only or with an
// on-device traceback; per-nucleotide hard constraints ('x' '<' '>') and Deigan stacking pseudo-energies folded in.
//
// Replaces the r background folds per window of energies()/rna_folder (ScanFoldFunctions.py:774-789,805-814)
// -- more than 99 % of all fold arithmetic of a scan -- and the native fold fc.mfe() of ScanFold.py:494-497,
// :512-513 (flag-only constraint lines) and :534-541 (Deigan).
//
// What changed against mfe2.cu: the <= 496 interior-loop candidates of a cell are no longer walked one by one.
// For generic loops (both sides >= 2 unpaired, not 2x2 / 2x3) of total size u the energy is
//     internal_loop[u] + min(MAX_NINIO, |u1-u2| * ninio) + mismatchI(outer) + mismatchI(inner),
// and all candidates of one u lie on ONE inner diagonal dd = d-2-u at consecutive positions.  With
// G = C + mismatchI(inner) stored per diagonal row, the near-symmetric candidates (|u1-u2| <= 4) are a fixed
// 5-tap (u even) or 4-tap (u odd) weighted stencil along the row, and every other candidate carries the same
// capped asymmetry term, so it only needs a range minimum of G over the row -- including the near ones in that
// range is harmless because the cap is an upper bound of their true term.  Per finished diagonal row the kernel
// stores the two stencils (NE, NO) and a sliding 8-minimum (M8); a cell then needs 1 + (1..4) loads per u
// instead of u-3.  Bulge and 1xn loops keep one load per candidate side: the bulge value (C + TerminalAU) and the 1xn
// value (C + mismatch1nI) of neighbouring cells share a 32-bit word, once in a copy indexed by the 5' end (loops
// with the unpaired bases on the 3' side) and once in a copy indexed by the 3' end (5' side), so that both loads have a
// lane-independent position.  With an odd word pitch / a row pitch of 31 (mod 32) words and the taps of disabled
// lanes redirected to the address of an enabled lane, every tap of the loop is one shared-memory wavefront (r01h: 16
// wavefronts for 9 loads, r01j: 7 for 7).
//
// Work split: the CTA walks the anti-diagonals two at a time (pairs d0, d0+1 with d0 odd) with ONE barrier per pair.
// Phase k (pair d0 = 5 + 2k) runs these mutually independent work units, each for one warp:
//   S   finalises C of the pair: the partial minima left by earlier phases plus the terms that need the previous
//       pair (stack, bulge of one, multiloop closing), then the derived rows G, NE, NO, M8, the bulge / 1xn words
//   F   the multiloop matrix FML of the PREVIOUS pair (d0-2, d0-1): it needs that pair's finished C rows
//   T   split minima of tile diagonal d0+1 (2x2 tiles; they only read FML of diagonals <= d0-3)
//   P   table-driven terms of the NEXT pair (d0+2, d0+3) that only read rows <= d0-1 (1x1, 2x1, 2x2, 2x3, hairpin,
//       generic 2x4 / 3x3 / 4x2 and the ends of sizes 9, 10): lane = pairable cell of a compacted list chunk
//   C   interior loops of size >= 2 of the next pair: one warp pass per pairable cell, lane = loop size
//   L   lists of the pairable cells of diagonals d0+4, d0+5
// so the only chain from pair to pair is S -> barrier -> S; everything else has a phase of slack.  (The first version
// had two barrier-separated phases per pair; late diagonals, which have fewer units than warps, paid two latency
// floors per pair.)
// int16 storage is exact as long as no stored energy drops below LOW16; a fold that does is flagged and redone
// by the int32 kernel (mfe.cu) in the same stream, so results never depend on which kernel ran.
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "device_common.cuh"

namespace sfb {
namespace {

constexpr int INF16 = 16000;
constexpr int TABLE_ENV16 = 2000;   // |table entry| the int16 arithmetic accepts (DESIGN §2)
constexpr int FIN16 = 4000;
constexpr int LOW16 = -12000;
constexpr int R32 = 32;  // ring depth of the rows read by loops of size <= 30 (written after the diagonal pair)
constexpr int R16 = 16;  // ring depth of raw C / pair type / G (read for small loops only)
constexpr int SEG = 25;  // row elements finished per warp pass in phase S (32 lanes - 7 halo lanes of the 8-minimum)

struct alignas(16) Tab3 {
    short stack[64], mmI[200], mm1n[200], mm23[200], mmH[200];
    short mlclose[200];        // mismatchM + TerminalAU + MLintern + MLclosing (closing pair of a multiloop)
    short mlstem[8 * 36];      // [type][5' code][3' code], code 5 = no neighbour: E_MLstem
    short ext[8 * 36];         // E_ExtLoop likewise
    short tAU[8];
    short bulge1;              // bulge[1]
    short il5_ninio;           // internal_loop[5] + ninio   (2x3 loops)
    short MLbase;
    short w1, w2, w3, w4;      // min(MAX_NINIO, k * ninio)
    short pad;
    unsigned char ptype[36];   // pair type of codes a*6+b (code 5 = sentinel)
    unsigned char rtype[8];
};

__constant__ int c3_il[32];     // internal_loop[u]                       (stencil rows already carry the asymmetry)
__constant__ int c3_cap[32];    // internal_loop[u] + MAX_NINIO
__constant__ int c3_size1[32];  // 1xn loops of total size u
__constant__ int c3_sizeB[32];  // bulge[u]
__constant__ int c3_sG6[4];     // generic loops of size 6: (2,4) (3,3) (4,2)
Tab3 *g_dtab3 = nullptr;
bool g_mfe3_ok = false;

constexpr int BIG = 1 << 20;  // size term of a disabled tap: the sum never wins whatever the load returns


// shared-memory accesses by 32-bit byte address: the interior-loop cell pass keeps one byte address per tap (row and
// offset folded in once per diagonal) and adds the cell's scaled index -- one integer instruction per load instead of the
// multiply-add + add the compiler emits when it rematerialises row * pitch + i per cell
__device__ __forceinline__ int lds_s16(unsigned a) {
    int v;
    asm volatile("ld.shared.s16 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ unsigned lds_u32(unsigned a) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ int4 lds_v4(unsigned a) {
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_u16(unsigned a, int v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((short)v));
}

template <int P, bool FMG = false>
struct Smem3 {
    static constexpr int KSM = FMG ? 4 : 2;   // copies of the split-minimum ring
    // ring pitch in shorts: PR/2 words = 31 (mod 32), so lane U reading row (c-U) at offset a*U (a = 0, 1/2, 1) lands in
    // bank (1+a/2)*U: the 32 taps of one warp load hit 32 different banks
    static constexpr int PR = P <= 64 ? P + 2 : ((P + 2 + 63) / 64) * 64 - 2;   // small windows: shared memory first
    static constexpr int PRW = (P + 3) | 1;   // pitch (32-bit words) of the paired bulge / 1xn rows: odd
    Tab3 tb;
    // ring rows and the square FML matrix, INF-initialised per fold; ne.. doubles as the staging area of C for
    // the exterior loop
    short ne[R32 * PR], no[R32 * PR], m8[R32 * PR];
    unsigned rpa[R32 * PRW];  // [row][p]: lo = C + TerminalAU of cell (p, p+dd), hi = C + mismatch1nI of cell (p+1, ..)
    unsigned rpq[R32 * PRW];  // [row][q]: lo = C + TerminalAU of cell (q-dd, q), hi = C + mismatch1nI of cell (.., q-1)
    short g[R16 * PR];
    short rc[R16 * PR];
    short fm[FMG ? 8 : P * P];   // fm[a][b]: FML[a,b] for b > a (row = 5' end), FML[b,a] for b < a (row = 3' end);
                                 // FMG: the matrix sits behind the scratch row in global memory instead
    short decp[KSM * 8 * PR];   // split minima of the last 8 diagonals, one copy per k part
    short partc[4 * PR], parts[4 * PR];   // partial minima by diagonal & 3: loops of size >= 2 / everything else
    short f5[P + 8];
    static constexpr int LP = P;              // list pitch (entries): a diagonal has fewer than P cells
    alignas(16) int list[(4 * LP + 16) * 4];     // per pairable cell: i, mismatchI / mismatch1nI / TerminalAU term of the
                                                 // closing pair; the traceback stack of the natives reuses it
    unsigned char ctx[R16 * PR];
    unsigned char sx[P + 8];   // sx[k+1] = code of nucleotide k, sx[0] = sx[W+1] = 5
    unsigned char sx5[P + 8], sx3[P + 8];   // the same, 5 (never pairs) where hard constraints forbid the nucleotide
                                            // as 5' / 3' partner ('x' both, '>' 5', '<' 3')
    alignas(16) int cnt[4];   // pairable cells of the diagonals d with d & 3 = slot (0 beyond the last diagonal)
    int wq[2];                // FMG: work-queue heads of the current / next phase (units are handed out dynamically)
    short scp[P + 8];   // soft constraints: scp[k] = sc[k] + sc[k+1] (0-based), the stack (i,j)-(i+1,j-1) adds scp[i] + scp[j-1]
    int minv[32];
    int fbest[32];   // per-length partial minima of an exterior-loop round (8 lengths x up to 4 slices)
    alignas(8) int stepinfo[(P / 2 + 4) * 2];    // per diagonal pair: unit counts of the phase (fold independent)
};

__host__ __device__ __forceinline__ int tri4(int d, int W) {  // first cell of diagonal d in the d >= 4 triangle
    return (d - 4) * W - ((d - 1) * d / 2 - 6);
}

// work units the split loop of tile diagonal D is cut into (long diagonals have few tiles: their k range is
// split over the lanes of one warp instead)
// FMG: the multiloop matrix lives in global memory (windows above 200 nt): its loads have L2 latency, so long split loops
// are cut in four whatever the number of tiles
__host__ __device__ __forceinline__ int ksplit(int D, int W, bool fmg = false) {
    if (fmg) return D >= 71 ? 4 : (D >= 36 ? 2 : 1);
    return (D < 36 || (W - 1 - D) / 2 + 1 <= 16) ? 1 : 2;
}

__device__ int hairpin_special3(const MfeTables *T, const Tab3 &tb, const unsigned char *sx, int i, int j, int type) {
    // loops of 3, 4 and 6 nucleotides: tabulated tri- / tetra- / hexaloops (SURVEY A.2); sx is offset by one
    const int u = j - i - 1;
    int e = T->hairpin_len[u];
    auto key = [&](int n) {
        int k = 0, mul = 1;
        for (int t = 0; t < n; t++) {
            k += sx[i + 1 + t] * mul;
            mul *= 5;
        }
        return k;
    };
    if (u == 4) {
        const int k = key(6);
        for (int t = 0; t < T->n_tetra; t++)
            if (T->tetra_key[t] == k) return T->tetra_e[t];
    } else if (u == 6) {
        const int k = key(8);
        for (int t = 0; t < T->n_hexa; t++)
            if (T->hexa_key[t] == k) return T->hexa_e[t];
    } else if (u == 3) {
        const int k = key(5);
        for (int t = 0; t < T->n_tri; t++)
            if (T->tri_key[t] == k) return T->tri_e[t];
        return e + tb.tAU[type];
    }
    return e + tb.mmH[(type * 5 + sx[i + 2]) * 5 + sx[j]];
}


// full interior-loop energy, all classes (traceback only; SURVEY A.2)
__device__ int e_intloop3(const MfeTables *T, int n1, int n2, int type, int t2, int si1, int sj1, int sp1, int sq1) {
    const int nl = max(n1, n2), ns = min(n1, n2);
    const int au = T->TerminalAU;
    if (nl == 0) return T->stack[type][t2];
    if (ns == 0) {
        int e = T->bulge[nl];
        if (nl == 1)
            e += T->stack[type][t2];
        else
            e += (type > 2 ? au : 0) + (t2 > 2 ? au : 0);
        return e;
    }
    if (ns == 1) {
        if (nl == 1) return T->int11[type][t2][si1][sj1];
        if (nl == 2) return n1 == 1 ? T->int21[type][t2][si1][sq1][sj1] : T->int21[t2][type][sq1][si1][sp1];
        return T->internal_loop[nl + 1] + min(T->max_ninio, (nl - ns) * T->ninio) + T->mismatch1nI[type][si1][sj1] +
               T->mismatch1nI[t2][sq1][sp1];
    }
    if (ns == 2) {
        if (nl == 2) return T->int22[type][t2][si1][sp1][sq1][sj1];
        if (nl == 3) return T->internal_loop[5] + T->ninio + T->mismatch23I[type][si1][sj1] + T->mismatch23I[t2][sq1][sp1];
    }
    return T->internal_loop[nl + ns] + min(T->max_ninio, (nl - ns) * T->ninio) + T->mismatchI[type][si1][sj1] +
           T->mismatchI[t2][sq1][sp1];
}

// Traceback by one warp in the candidate order of SURVEY A.4 (the same order as mfe.cu's serial traceback): the
// control flow is warp-uniform, every candidate search is spread over the lanes and the first match in order wins.
// cx: C + exterior stem term by diagonal (the F5 staging area); pt: 1-based partner, 0 = unpaired.
template <int P, bool FMG, class SMT>
__device__ bool traceback3(SMT &sm, const short *fm, const MfeTables *T, const short *cx, short *pt, int W, int lane) {
    const Tab3 &tb = sm.tb;
    const unsigned char *sx = sm.sx;
    const unsigned full = 0xffffffffu;
    static_assert(sizeof(sm.list) >= 3 * (P + 8) * sizeof(int), "the traceback stack lives in the list area");
    int *stk = reinterpret_cast<int *>(sm.list);
    auto ptype = [&](int a, int b) { return (int)tb.ptype[sx[a + 1] * 6 + sx[b + 1]]; };
    auto CC = [&](int i, int j) {
        const int v = cx[tri4(j - i, W) + i];
        return v >= FIN16 ? INF : v - tb.ext[ptype(i, j) * 36 + sx[i] * 6 + sx[j + 2]];
    };
    auto MM = [&](int i, int j) {
        if (j - i <= TURN) return INF;
        int v;
        if constexpr (FMG) v = __ldcg(fm + i * P + j);
        else v = fm[i * P + j];
        return v >= FIN16 ? INF : v;
    };
    for (int k = lane; k < W; k += 32) pt[k] = 0;
    int sp = 1;
    if (lane == 0) {
        stk[0] = 0;
        stk[1] = W - 1;
        stk[2] = 0;
    }
    __syncwarp();
    while (sp > 0) {
        sp--;
        int i = stk[3 * sp], j = stk[3 * sp + 1];
        const int ml = stk[3 * sp + 2];
        __syncwarp();
        bool have_pair = false;
        if (j < i + TURN + 1) continue;
        const int fij = ml ? MM(i, j) : (int)sm.f5[j + 1];
        const int mij1 = MM(i, j - 1);
        const int fi = ml ? (mij1 < INF ? mij1 + tb.MLbase : INF) : (int)sm.f5[j];
        auto push = [&](int a, int b, int c) {
            if (lane == 0) {
                stk[3 * sp] = a;
                stk[3 * sp + 1] = b;
                stk[3 * sp + 2] = c;
            }
            sp++;
        };
        if (fij == fi) {
            push(i, j - 1, ml);
            __syncwarp();
            continue;
        }
        if (ml == 0) {
            int kf = -1;
            for (int k0 = j - TURN - 1; k0 >= 0 && kf < 0; k0 -= 32) {
                const int k = k0 - lane;
                bool hit = false;
                if (k >= 0) {
                    const int ckj = CC(k, j);
                    hit = ckj < INF && fij == tb.ext[ptype(k, j) * 36 + sx[k] * 6 + sx[j + 2]] + ckj + sm.f5[k];
                }
                const unsigned m = __ballot_sync(full, hit);
                if (m) kf = k0 - (__ffs(m) - 1);
            }
            if (kf < 0) return false;
            push(0, kf - 1, 0);
            i = kf;
            have_pair = true;
        } else {
            const int mi1j = MM(i + 1, j);
            if (mi1j < INF && mi1j + tb.MLbase == fij) {
                push(i + 1, j, 1);
                __syncwarp();
                continue;
            }
            const int cij = CC(i, j);
            if (cij < INF && fij == cij + tb.mlstem[ptype(i, j) * 36 + sx[i] * 6 + sx[j + 2]]) {
                have_pair = true;
            } else {
                int kf = -1;
                for (int k0 = i + 1 + TURN; k0 <= j - 2 - TURN && kf < 0; k0 += 32) {
                    const int k = k0 + lane;
                    bool hit = false;
                    if (k <= j - 2 - TURN) {
                        const int a = MM(i, k), b = MM(k + 1, j);
                        hit = a < INF && b < INF && fij == a + b;
                    }
                    const unsigned m = __ballot_sync(full, hit);
                    if (m) kf = k0 + __ffs(m) - 1;
                }
                if (kf < 0) return false;
                push(i, kf, 1);
                push(kf + 1, j, 1);
                __syncwarp();
                continue;
            }
        }
        while (have_pair) {
            if (lane == 0) {
                pt[i] = (short)(j + 1);
                pt[j] = (short)(i + 1);
            }
            const int type = ptype(i, j);
            const int cij = CC(i, j);
            if (cij == hairpin_special3(T, tb, sx, i, j, type)) break;
            bool traced = false;
            const int pmax = min(j - 2 - TURN, i + MAXLOOP + 1);
            for (int p = i + 1; p <= pmax && !traced; p++) {
                int minq = j - i + p - MAXLOOP - 2;
                if (minq < p + 1 + TURN) minq = p + 1 + TURN;
                const int q = j - 1 - lane;   // at most 31 candidates per p
                bool hit = false;
                if (q >= minq) {
                    const int cpq = CC(p, q);
                    if (cpq < INF) {
                        const int t2 = tb.rtype[ptype(p, q)];
                        int e = e_intloop3(T, p - i - 1, j - q - 1, type, t2, sx[i + 2], sx[j], sx[p], sx[q + 2]);
                        if (p == i + 1 && q == j - 1) e += sm.scp[i] + sm.scp[j - 1];   // Deigan: stacked pairs only
                        hit = cij == e + cpq;
                    }
                }
                const unsigned m = __ballot_sync(full, hit);
                if (m) {
                    j = j - 1 - (__ffs(m) - 1);
                    i = p;
                    traced = true;
                }
            }
            if (traced) continue;
            const int en = cij - tb.mlclose[(tb.rtype[type] * 5 + sx[j]) * 5 + sx[i + 2]];
            int kf = -1;
            for (int k0 = i + 2 + TURN; k0 < j - 2 - TURN && kf < 0; k0 += 32) {
                const int k = k0 + lane;
                bool hit = false;
                if (k < j - 2 - TURN) {
                    const int a = MM(i + 1, k), b = MM(k + 1, j - 1);
                    hit = a < INF && b < INF && en == a + b;
                }
                const unsigned m = __ballot_sync(full, hit);
                if (m) kf = k0 + __ffs(m) - 1;
            }
            if (kf < 0) return false;
            push(i + 1, kf, 1);
            push(kf + 1, j - 1, 1);
            break;
        }
        __syncwarp();
    }
    return true;
}

template <int P, int NW, int OCC, bool FMG>
__global__ void __launch_bounds__(NW * 32, OCC)
mfe3_kernel(MfeLaunch L, const MfeTables *__restrict__ T, const Tab3 *__restrict__ gtab) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using SM = Smem3<P, FMG>;
    SM &sm = *reinterpret_cast<SM *>(smem_raw);
    constexpr int NT = NW * 32, PR = SM::PR;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const unsigned full = 0xffffffffu;
    {
        const int *src = reinterpret_cast<const int *>(gtab);
        int *dst = reinterpret_cast<int *>(&sm.tb);
        static_assert(sizeof(Tab3) % 4 == 0, "Tab3 is copied as 32-bit words");
        for (int k = tid; k < (int)(sizeof(Tab3) / 4); k += NT) dst[k] = src[k];
    }
    const Tab3 &tb = sm.tb;
    const unsigned char *sx = sm.sx;
    const int W = L.W;
    constexpr int LP = SM::LP;
    const int npairs = (W - TURN) / 2 + 1;   // phases: pairs d0 = 5, 7, .. while d0 - 2 < W (F runs one pair behind)
    for (int st = tid; st < npairs; st += NT) {
        const int d0 = TURN + 2 + 2 * st;
        const int nseg0 = d0 < W ? (W - d0 + SEG - 1) / SEG : 0, nseg1 = d0 + 1 < W ? (W - d0 - 1 + SEG - 1) / SEG : 0;
        const int nF = d0 - 2 < W ? (W - (d0 - 2) + 30) / 31 : 0;
        const int D = d0 + 1;
        const int ntile = D <= W - 1 ? (W - 1 - D) / 2 + 1 : 0;
        const int KS = ksplit(D, W, FMG), ksh = KS == 4 ? 2 : KS >> 1 /* log2 of 1, 2, 4 */;
        const int kwsh = ntile > 16 ? 0 : (ntile > 8 ? 1 : 2), TPW = 32 >> kwsh;   // k parts inside a warp
        const int nT = ((ntile + TPW - 1) >> (5 - kwsh)) << ksh;
        reinterpret_cast<int2 *>(sm.stepinfo)[st] =
            make_int2(nseg0 | ((nseg0 + nseg1) << 8) | (nF << 16), ntile | (ksh << 8) | (kwsh << 12) | (nT << 16));
    }
    short *gC = reinterpret_cast<short *>(L.gscratch) + (size_t)blockIdx.x * L.gscratch_per_cta;
    auto ldfm = [&](const short *q) -> short {   // FMG: from L2 (written by this CTA in an earlier phase)
        if constexpr (FMG) return __ldcg(q);
        else return *q;
    };
    // the multiloop matrix: shared memory, or (FMG) the P x P shorts behind the scratch row of this CTA
    short *const fm = FMG ? gC + (((size_t)tri4(W, W) + 63) & ~(size_t)63) : sm.fm;
    const short *smb = sm.ne;   // every tap address below is an offset (in shorts) from here
    constexpr int PRW = SM::PRW;
    constexpr int O_NE = 0, O_NO = R32 * PR, O_M8 = 2 * R32 * PR;   // in shorts from smb
    static_assert(offsetof(SM, no) - offsetof(SM, ne) == 2 * O_NO && offsetof(SM, m8) - offsetof(SM, ne) == 2 * O_M8,
                  "tap offsets follow the member order");

    // ---- per-lane loop size U = lane: size terms of its nine taps (see the header); BIG disables a tap
    const int U = lane;
    const bool uok = U <= MAXLOOP;
    const int cSB = (uok && U >= 2) ? c3_sizeB[U] : BIG;
    const int cS1 = (uok && U >= 4) ? c3_size1[U] : BIG;
    const int cA = (uok && U >= 7) ? c3_il[U] : BIG;        // generic loops of size 6 and the two end candidates of
    const int cB10 = (uok && U >= 11) ? c3_cap[U] : BIG;    // sizes 9, 10 are table-driven terms (do_special)
    const int cB18 = (uok && U > 19) ? c3_cap[U] : BIG;
    const int cB26 = (uok && U > 27) ? c3_cap[U] : BIG;
    const int cC = (uok && U > 11) ? c3_cap[U] : BIG;
    // a disabled tap reads the address of an enabled lane (same word: a broadcast, never a bank conflict)
    // rows d-2, d-3 are being written in the same phase: the (disabled) lanes 0, 1 read the rows of lanes 2, 3 instead.
    // The three range-minimum taps (offsets 10, 18, 26 of the M8 row) do the same with the rows of lanes 11, 20, 28: an
    // enabled tap never leaves its row (row d-2-U has W-d+2+U entries), while a disabled one at its own row could run
    // past a short row's end into the ring row unit S is writing in the same phase (racecheck r01: mfe3.cu:530 / :718).
    const int UB = U < 2 ? U + 2 : (U > MAXLOOP ? MAXLOOP : U);
    const int UA = U < 7 ? U + 8 : (U > MAXLOOP ? MAXLOOP - 1 : U);
    const int UC = U < 12 ? U + 12 : (U > MAXLOOP ? MAXLOOP : U);
    const int UB10 = U < 11 ? 11 : (U > MAXLOOP ? MAXLOOP : U), UB18 = U < 20 ? 20 : (U > MAXLOOP ? MAXLOOP : U);
    const int UB26 = U < 28 ? 28 : (U > MAXLOOP ? MAXLOOP : U);
    const int kA = ((UA & 1) ? O_NO : O_NE) + 3 + (UA >> 1), kC = O_M8 + UC - 1;
    const int g6a = c3_sG6[0], g6b = c3_sG6[1], g6c = c3_sG6[2], g9 = c3_cap[9], g10 = c3_cap[10];

    // compacted list of the pairable cells of diagonal d with the closing-pair terms (one warp) -> slot d & 3
    auto build_list = [&](int d) {
        const int ncells = W - d, slot = d & 3;
        constexpr int NCH = (P + 31) / 32;
        // pair types of every chunk of 32 cells first (independent loads), then the compaction chunk by chunk
        int tt[NCH];
#pragma unroll
        for (int k = 0; k < NCH; k++) {
            const int i = k * 32 + lane;
            tt[k] = i < ncells ? tb.ptype[sm.sx5[i + 1] * 6 + sm.sx3[i + d + 1]] : 0;
        }
        int nl = 0;
#pragma unroll
        for (int k = 0; k < NCH; k++) {
            if (k * 32 < ncells) {   // warp-uniform
                const int i = k * 32 + lane, t = tt[k];
                const unsigned m = __ballot_sync(full, t != 0);
                if (t) {
                    const int mi = (t * 5 + sx[i + 2]) * 5 + sx[i + d];
                    const int4 en = make_int4(i, tb.mmI[mi], tb.mm1n[mi], tb.tAU[t]);
                    reinterpret_cast<int4 *>(sm.list)[slot * LP + nl + __popc(m & ((1u << lane) - 1))] = en;
                }
                nl += __popc(m);
            }
        }
        if (lane == 0) sm.cnt[slot] = nl;
    };
    // split minimum of cell (xi, d): which tile diagonal produced it decides how many partials exist
    auto decof = [&](int d, int xi) {
        if (d < 2 * TURN + 3) return INF16;
        const int Dsrc = (d & 1) ? ((xi & 1) ? d + 1 : d - 1) : d;
        const int ks = ksplit(Dsrc, W, FMG);
        int v = sm.decp[(d & 7) * PR + xi];
        for (int kp = 1; kp < ks; kp++) v = min(v, (int)sm.decp[(kp * 8 + (d & 7)) * PR + xi]);
        return v;
    };
    // unit P: table-driven terms of the pairable cells of diagonal d, list chunk c (lane = cell), that only read rows
    // <= d-4; stack, bulge of one and multiloop closing are added when the cell is finalised (unit S)
    auto unit_P = [&](int d, int c) {
        const int slot = d & 3, n = sm.cnt[slot];
        const int idx = c * 32 + lane;
        const bool active = idx < n;
        const int i = active ? sm.list[(slot * LP + idx) * 4] : 0;
        const int j = i + d;
        const int type = tb.ptype[sx[i + 1] * 6 + sx[j + 1]];
        const int si1 = sx[i + 2], sj1 = sx[j];
        const int mi = (type * 5 + si1) * 5 + sj1;
        int aT = INF16;
        auto inner = [&](int u1, int u2, int &cc, int &t2, int &sp1, int &sq1) {
            const int dd = d - 2 - u1 - u2, p = i + 1 + u1, q = j - 1 - u2;
            const bool ok = dd > TURN;
            cc = ok ? sm.rc[(dd & (R16 - 1)) * PR + p] : INF16;
            t2 = ok ? sm.ctx[(dd & (R16 - 1)) * PR + p] : 0;
            sp1 = sx[p];       // S[p-1]
            sq1 = sx[q + 2];   // S[q+1]
        };
        int cc, t2, sp1, sq1;
        {
            inner(1, 1, cc, t2, sp1, sq1);
            aT = min(aT, cc + __ldg(&T->int11[type][t2][si1][sj1]));
            int eh = __ldg(&T->hairpin_len[d - 1]) + tb.mmH[mi];
            if (d <= 7 && active) eh = hairpin_special3(T, tb, sx, i, j, type);
            aT = min(aT, eh);
            inner(1, 2, cc, t2, sp1, sq1);
            aT = min(aT, cc + __ldg(&T->int21[type][t2][si1][sq1][sj1]));
            inner(2, 1, cc, t2, sp1, sq1);
            aT = min(aT, cc + __ldg(&T->int21[t2][type][sq1][si1][sp1]));
            inner(2, 2, cc, t2, sp1, sq1);
            aT = min(aT, cc + __ldg(&T->int22[type][t2][si1][sp1][sq1][sj1]));
            inner(2, 3, cc, t2, sp1, sq1);
            aT = min(aT, cc + tb.il5_ninio + tb.mm23[mi] + tb.mm23[(t2 * 5 + sq1) * 5 + sp1]);
            inner(3, 2, cc, t2, sp1, sq1);
            aT = min(aT, cc + tb.il5_ninio + tb.mm23[mi] + tb.mm23[(t2 * 5 + sq1) * 5 + sp1]);
            // generic loops the stencil / range rows do not cover: 2x4 3x3 4x2 and the two ends of sizes 9, 10
            auto grow = [&](int dd, int p) { return dd > TURN ? (int)sm.g[(dd & (R16 - 1)) * PR + p] : INF16; };
            int aG = min(grow(d - 8, i + 3) + g6a, min(grow(d - 8, i + 4) + g6b, grow(d - 8, i + 5) + g6c));
            aG = min(aG, min(grow(d - 11, i + 3), grow(d - 11, i + 8)) + g9);
            aG = min(aG, min(grow(d - 12, i + 3), grow(d - 12, i + 9)) + g10);
            aT = min(aT, aG + tb.mmI[mi]);
        }
        if (active) sm.parts[slot * PR + i] = (short)min(aT, INF16);
    };

    int minv = 0;   // smallest stored energy of the fold (int16 range check)

    // unit S: 25 row elements of diagonal d -- C from the partial minima and the terms that need the previous pair,
    // then the derived rows (warp shuffles along the row; lanes 0..6 are the halo of the sliding minimum)
    auto unit_S = [&](int d, int sg) {
        const int ncells = W - d;
        const int x = sg * SEG - 7 + lane;
        const bool valid = x >= 0 && x < ncells;
        const int i = valid ? x : 0, j = i + d;
        // every load whose address does not depend on the pair type is issued before the type is known, the table lookups
        // that do in one second round: three dependent shared-memory round trips instead of five (a lane that is no pair or
        // sits outside the row reads valid but meaningless entries and is masked)
        const int c5 = sm.sx5[i + 1], c3 = sm.sx3[j + 1];
        const int pc = sm.partc[(d & 3) * PR + i], ps = sm.parts[(d & 3) * PR + i];
        const int o2 = ((d - 2) & (R16 - 1)) * PR + i + 1, o3 = ((d - 3) & (R16 - 1)) * PR + i + 1;
        const int rc2 = sm.rc[o2], cx2 = sm.ctx[o2];
        const int rc3a = sm.rc[o3], cx3a = sm.ctx[o3], rc3b = sm.rc[o3 + 1], cx3b = sm.ctx[o3 + 1];
        const int dm = decof(d - 2, i + 1);   // multiloop closed by (i,j)
        const int si0 = sx[i], si2 = sx[i + 2], sj0 = sx[j], sj2 = sx[j + 2];
        int scs = 0;
        if (L.sc) scs = sm.scp[i] + sm.scp[j - 1];   // Deigan pseudo-energy of the stack (kernel-uniform branch)
        const int t = valid ? tb.ptype[c5 * 6 + c3] : 0;
        const int t2 = tb.rtype[t];
        const int st2 = tb.stack[t * 8 + cx2], st3a = tb.stack[t * 8 + cx3a], st3b = tb.stack[t * 8 + cx3b];
        const int mlc = tb.mlclose[(t2 * 5 + sj0) * 5 + si2];
        const int m2 = (t2 * 5 + sj2) * 5 + si0;
        const int xI = tb.mmI[m2], x1n = tb.mm1n[m2], xAU = tb.tAU[t2];
        int e = min(pc, ps);
        if (d - 2 > TURN) e = min(e, rc2 + st2 + scs);                            // stack: inner pair (i+1, j-1)
        if (d - 3 > TURN) e = min(e, min(rc3a + st3a, rc3b + st3b) + tb.bulge1);   // bulge of one: (i+1, j-2) and (i+2, j-1)
        e = min(e, dm + mlc);
        if (!t || e >= FIN16) e = INF16;
        int vg = INF16, v1 = INF16, vb = INF16;
        if (t && i > 0 && j < W - 1 && e < FIN16) {
            vg = e + xI;
            v1 = e + x1n;
            vb = e + xAU;
        }
        const int g1 = __shfl_up_sync(full, vg, 1), g2 = __shfl_up_sync(full, vg, 2);
        const int g3 = __shfl_up_sync(full, vg, 3), g4 = __shfl_up_sync(full, vg, 4);
        const int ne = min(g2, min(min(g1, g3) + tb.w2, min(vg, g4) + tb.w4));
        const int no = min(min(g1, g2) + tb.w1, min(vg, g3) + tb.w3);
        int m8 = min(vg, g1);
        m8 = min(m8, __shfl_up_sync(full, m8, 2));
        m8 = min(m8, __shfl_up_sync(full, m8, 4));
        if (valid && lane >= 7) {
            minv = min(minv, e);
            const int o16 = (d & (R16 - 1)) * PR + i, o32 = (d & (R32 - 1)) * PR + i;
            sm.rc[o16] = (short)e;
            sm.ctx[o16] = (unsigned char)t2;
            sm.g[o16] = (short)vg;
            {   // bulge | 1xn pairs: 16-bit halves of the 5'-indexed and the 3'-indexed copy
                short *wa = reinterpret_cast<short *>(sm.rpa) + 2 * ((d & (R32 - 1)) * PRW + i);
                short *wq = reinterpret_cast<short *>(sm.rpq) + 2 * ((d & (R32 - 1)) * PRW + j);
                wa[0] = (short)vb;
                if (i > 0) wa[-1] = (short)v1;
                wq[0] = (short)vb;
                wq[3] = (short)v1;
            }
            sm.ne[o32] = (short)ne;
            sm.no[o32] = (short)no;
            sm.m8[o32] = (short)m8;
            gC[tri4(d, W) + i] = (short)(e < FIN16 ? e + tb.ext[t * 36 + sx[i] * 6 + sx[j + 2]] : INF16);
        }
    };

    // unit F: 31 cells of the multiloop matrix of diagonals dA, dA+1 (the neighbour on dA comes by shuffle)
    auto unit_F = [&](int dA, int u) {
        const int nc0 = dA > TURN ? W - dA : 0, nc1 = dA + 1 < W ? W - dA - 1 : 0;
        const int x = u * 31 + lane;
        const bool v0 = x < nc0;
        const int xx = v0 ? x : max(nc0 - 1, 0);
        auto stemof = [&](int d, int xi) {
            const int o16 = (d & (R16 - 1)) * PR + xi;
            const int e = sm.rc[o16];
            const int t = tb.rtype[sm.ctx[o16]];
            return e < FIN16 ? e + tb.mlstem[t * 36 + sx[xi] * 6 + sx[xi + d + 2]] : INF16;
        };
        // the loads of both diagonals first (clamped positions, masked afterwards): the second cell only waits for the first
        // one's value, not for its own operands
        const int x1c = min(x, max(nc1 - 1, 0));
        const int s0 = min(decof(dA, xx), stemof(dA, xx));
        const int s1 = min(decof(dA + 1, x1c), stemof(dA + 1, x1c));
        int m0 = INF16;
        if (nc0 > 0) {
            m0 = s0;
            if (dA - 1 > TURN)
                m0 = min(m0, min((int)ldfm(fm + (xx + 1) * P + xx + dA), (int)ldfm(fm + xx * P + xx + dA - 1)) + tb.MLbase);
            if (m0 >= FIN16) m0 = INF16;
            if (v0) {
                minv = min(minv, m0);
                fm[x * P + x + dA] = (short)m0;
                fm[(x + dA) * P + x] = (short)m0;
            }
        }
        const int m0n = __shfl_down_sync(full, m0, 1);
        if (lane < 31 && x < nc1) {
            const int d = dA + 1;
            int m1 = min(s1, min(m0, m0n) + tb.MLbase);
            if (m1 >= FIN16) m1 = INF16;
            minv = min(minv, m1);
            fm[x * P + x + d] = (short)m1;
            fm[(x + d) * P + x] = (short)m1;
        }
    };

    // unit T: 2x2 tiles (i, i+1) x (j, j+1), i and j even, j - i = D: all four split minima share their operands; both
    // operand pairs are one aligned 32-bit load from the square matrix.  Lanes = tiles x k parts; further k parts are
    // separate units (partials in decp).  k = i+4 .. j-4 only touches FML of diagonals <= D-4.
    auto unit_T = [&](int D, int q, int ntile, int ksh, int kwsh) {
        const int KS = 1 << ksh, TPW = 32 >> kwsh;
        const int grp = q >> ksh, kp = q & (KS - 1);
        const int tl = grp * TPW + (lane & (TPW - 1)), kq = lane >> (5 - kwsh);
        const bool valid = tl < ntile;
        const int i = 2 * min(tl, ntile - 1), j = i + D;
        const int cntk = max(D - 7, 0);
        const int pidx = (kp << kwsh) + kq, psh = ksh + kwsh;
        const int k0 = i + 4 + ((cntk * pidx) >> psh), k1 = i + 4 + ((cntk * (pidx + 1)) >> psh);
        unsigned acc0 = INF16 * 65537u, acc1 = INF16 * 65537u;
        if constexpr (FMG) {
            // Global matrix: the lanes of a k part sweep the SAME rows, so a warp load is one contiguous row segment
            // (the per-tile windows k = i+4 .. j-4 start two rows apart from tile to tile; with each lane on its own
            // row a load touched 32 sectors).  The sweep covers the union of the windows; a lane outside its own
            // window contributes INF.
            const int ltl = lane & (TPW - 1);
            const int ibase = 2 * grp * TPW;                 // i of the group's first tile
            const int span = cntk + 2 * (TPW - 1);
            const int s0 = (span * pidx) >> psh, s1 = min((span * (pidx + 1)) >> psh, P - 5 - ibase);   // rows stay inside
            const unsigned *pa = reinterpret_cast<const unsigned *>(fm + (ibase + 4 + s0) * P + i);
            const unsigned *pb = reinterpret_cast<const unsigned *>(fm + (ibase + 5 + s0) * P + j);
            const unsigned infp = INF16 * 65537u;
            int kk = s0;
            constexpr int UNR = 8;
            for (; kk + UNR - 1 < s1; kk += UNR, pa += UNR * (P / 2), pb += UNR * (P / 2)) {
                unsigned a[UNR], b[UNR];
#pragma unroll
                for (int z = 0; z < UNR; z++) {
                    a[z] = __ldcg(pa + z * (P / 2));
                    b[z] = __ldcg(pb + z * (P / 2));
                }
#pragma unroll
                for (int z = 0; z < UNR; z++) {
                    const unsigned rel = (unsigned)(kk + z - 2 * ltl);
                    const unsigned av = rel < (unsigned)cntk ? a[z] : infp;
                    acc0 = __viaddmin_s16x2(av, __byte_perm(b[z], 0, 0x1010), acc0);
                    acc1 = __viaddmin_s16x2(av, __byte_perm(b[z], 0, 0x3232), acc1);
                }
            }
            for (; kk < s1; kk++, pa += P / 2, pb += P / 2) {
                const unsigned rel = (unsigned)(kk - 2 * ltl);
                const unsigned av = rel < (unsigned)cntk ? __ldcg(pa) : infp, b = __ldcg(pb);
                acc0 = __viaddmin_s16x2(av, __byte_perm(b, 0, 0x1010), acc0);
                acc1 = __viaddmin_s16x2(av, __byte_perm(b, 0, 0x3232), acc1);
            }
        } else {
            const unsigned *pa = reinterpret_cast<const unsigned *>(fm + k0 * P + i);
            const unsigned *pb = reinterpret_cast<const unsigned *>(fm + (k0 + 1) * P + j);
            int k = k0;
            for (; k + 3 < k1; k += 4, pa += 2 * P, pb += 2 * P) {
#pragma unroll
                for (int z = 0; z < 4; z++) {
                    const unsigned a = pa[z * (P / 2)], b = pb[z * (P / 2)];
                    acc0 = __viaddmin_s16x2(a, __byte_perm(b, 0, 0x1010), acc0);
                    acc1 = __viaddmin_s16x2(a, __byte_perm(b, 0, 0x3232), acc1);
                }
            }
            for (; k < k1; k++, pa += P / 2, pb += P / 2) {
                const unsigned a = pa[0], b = pb[0];
                acc0 = __viaddmin_s16x2(a, __byte_perm(b, 0, 0x1010), acc0);
                acc1 = __viaddmin_s16x2(a, __byte_perm(b, 0, 0x3232), acc1);
            }
        }
        if (kwsh >= 1) {
            acc0 = __vmins2(acc0, __shfl_xor_sync(full, acc0, 16));
            acc1 = __vmins2(acc1, __shfl_xor_sync(full, acc1, 16));
        }
        if (kwsh == 2) {
            acc0 = __vmins2(acc0, __shfl_xor_sync(full, acc0, 8));
            acc1 = __vmins2(acc1, __shfl_xor_sync(full, acc1, 8));
        }
        if (valid && kq == 0) {
            auto fin = [](int v) { return (short)(v >= FIN16 ? INF16 : v); };
            short *dp = sm.decp + kp * 8 * PR;
            dp[(D & 7) * PR + i] = fin((short)(acc0 & 0xffffu));
            dp[((D - 1) & 7) * PR + i + 1] = fin((int)acc0 >> 16);
            if (j + 1 < W) {
                dp[((D + 1) & 7) * PR + i] = fin((short)(acc1 & 0xffffu));
                dp[(D & 7) * PR + i + 1] = fin((int)acc1 >> 16);
            }
        }
    };

    for (int fold = blockIdx.x; fold < L.n_fold; fold += gridDim.x) {
        __syncthreads();
        // ---- prologue: sequence with sentinels, INF in every ring row and in the FML matrix
        for (int k = tid; k < W + 2; k += NT) {
            const bool edge = k == 0 || k == W + 1;
            const int code = edge ? 5 : L.seqs[(size_t)fold * W + k - 1];
            const char ch = (L.hc && !edge) ? (char)L.hc[(size_t)fold * W + k - 1] : '.';
            sm.sx[k] = (unsigned char)code;
            sm.sx5[k] = (unsigned char)((ch == 'x' || ch == '>') ? 5 : code);   // '>' : pairs upstream only (SURVEY A.5)
            sm.sx3[k] = (unsigned char)((ch == 'x' || ch == '<') ? 5 : code);   // '<' : pairs downstream only
        }
        {
            const int4 inf4 = make_int4(INF16 * 65537, INF16 * 65537, INF16 * 65537, INF16 * 65537);
            int4 *p = reinterpret_cast<int4 *>(sm.ne);
            constexpr int n16 = (int)((offsetof(SM, decp) - offsetof(SM, ne) + 15) / 16);   // a ragged tail spills
            for (int k = tid; k < n16; k += NT) p[k] = inf4;                                 // into decp (rewritten before use)
            for (int k = tid; k < 4 * PR; k += NT) sm.partc[k] = INF16;   // diagonals 4 .. 7 have no interior loops of size >= 2
            if constexpr (FMG) {
                int4 *q = reinterpret_cast<int4 *>(fm);
                for (int k = tid; k < P * P / 8; k += NT) q[k] = inf4;
            }
        }
        minv = 0;
        if (tid < 2) sm.wq[tid] = 0;
        for (int k = tid; k < W + 2; k += NT) {
            int v = 0;
            if (L.sc && k < W) {   // L.sc is 1-based: nucleotide k sits at index k + 1
                const int a = L.sc[(size_t)fold * (W + 1) + k + 1], b = k + 1 < W ? L.sc[(size_t)fold * (W + 1) + k + 2] : 0;
                v = a + b;
                if (abs(a) > 4000 || abs(b) > 4000) minv = LOW16 - 1;   // int16 cannot hold it: redo in int32
            }
            sm.scp[k] = (short)max(-8000, min(8000, v));
        }
        __syncthreads();
        // diagonals 4 .. 6: lists, hairpins (all they can close), then the rows of diagonal 4 and the lists of 7, 8
        if (warp < 3) build_list(TURN + 1 + warp);
        __syncthreads();
        {
            const int c4 = (sm.cnt[0] + 31) >> 5, c5 = (sm.cnt[1] + 31) >> 5, c6 = (sm.cnt[2] + 31) >> 5;
            for (int it = warp; it < c4 + c5 + c6; it += NW) {
                if (it < c4)
                    unit_P(TURN + 1, it);
                else if (it < c4 + c5)
                    unit_P(TURN + 2, it - c4);
                else
                    unit_P(TURN + 3, it - c4 - c5);
            }
        }
        __syncthreads();
        for (int u = warp; u < (W - TURN - 1 + SEG - 1) / SEG + 2; u += NW) {
            if (u < 2)
                build_list(TURN + 4 + u);   // slots 3 and 0: the list of diagonal 4 is no longer needed
            else
                unit_S(TURN + 1, u - 2);
        }
        __syncthreads();

        // ---- C (queue variant): interior loops of size >= 2 of the pairable cells c .. n-1 of diagonal d (d0+2 or d0+3;
        // rows <= d0-1): one cell per pass, lane = loop size U with its seven taps (see the header)
        auto unit_C = [&](int d, int c, int n) {
            const int slot = (d - 2 - UB) & (R32 - 1);
            const unsigned sb = (unsigned)__cvta_generic_to_shared(smb);
            const unsigned aA = sb + 2 * (kA + ((d - 2 - UA) & (R32 - 1)) * PR);
            const unsigned aB10 = sb + 2 * (O_M8 + 10 + ((d - 2 - UB10) & (R32 - 1)) * PR);
            const unsigned aB18 = sb + 2 * (O_M8 + 18 + ((d - 2 - UB18) & (R32 - 1)) * PR);
            const unsigned aB26 = sb + 2 * (O_M8 + 26 + ((d - 2 - UB26) & (R32 - 1)) * PR);
            const unsigned aC = sb + 2 * (kC + ((d - 2 - UC) & (R32 - 1)) * PR);
            const unsigned aR = (unsigned)__cvta_generic_to_shared(sm.rpa + slot * PRW + 1);       // inner pair (i+1, j-1-U) and 1xn neighbour
            const unsigned aL = (unsigned)__cvta_generic_to_shared(sm.rpq + slot * PRW + d - 1);   // inner pair (i+1+U, j-1) and 1xn neighbour
            const unsigned aP = (unsigned)__cvta_generic_to_shared(sm.partc + (d & 3) * PR);
            unsigned aLst = (unsigned)__cvta_generic_to_shared(reinterpret_cast<const int4 *>(sm.list) + (d & 3) * LP + c);
            int4 en = lds_v4(aLst);
            for (; c < n; c++) {
                const int i = en.x, eI = en.y, e1 = en.z, eB = en.w;
                aLst += 16;
                en = lds_v4(aLst);   // next entry (at most one past the list end: still inside sm.list)
                const unsigned i2 = 2 * i, i4 = 4 * i;
                const unsigned wr = lds_u32(aR + i4), wl = lds_u32(aL + i4);
                const int xa = lds_s16(aA + i2), xb10 = lds_s16(aB10 + i2), xb18 = lds_s16(aB18 + i2);
                const int xb26 = lds_s16(aB26 + i2), xc = lds_s16(aC + i2);
                const unsigned wm = __vmins2(wr, wl);
                const int xb = (int)(short)(wm & 0xffffu), x1 = (int)wm >> 16;
                int g = xa + cA;
                g = __viaddmin_s32(xb10, cB10, g);
                int g2 = xb18 + cB18;
                g2 = __viaddmin_s32(xb26, cB26, g2);
                g = __viaddmin_s32(xc, cC, g);
                const int aB = xb + cSB, a1 = x1 + cS1;
                int v = min(g, g2) + eI;
                v = __viaddmin_s32(a1, e1, v);
                v = __viaddmin_s32(aB, eB, v);
                v = __reduce_min_sync(full, v);
                if (lane == 0) sts_u16(aP + i2, v);   // <= INF16 + size and mismatch terms: fits
            }
        };

        for (int d0 = TURN + 2, ph = 0; d0 - 2 < W; d0 += 2, ph ^= 1) {
            const int2 si = reinterpret_cast<const int2 *>(sm.stepinfo)[(d0 - TURN - 2) >> 1];
            const int nseg0 = si.x & 255, nS = (si.x >> 8) & 255, nF = si.x >> 16;
            const int ntile = si.y & 255, ksh = (si.y >> 8) & 15, kwsh = (si.y >> 12) & 15, nT = si.y >> 16;
            const int n2 = sm.cnt[(d0 + 2) & 3], n3 = sm.cnt[(d0 + 3) & 3];   // (the other two slots are being rewritten)
            const int nch2 = (n2 + 31) >> 5, nP = nch2 + ((n3 + 31) >> 5);
            if constexpr (FMG) {
                // One CTA per SM and long split loops over L2: the units of a phase differ in length by an order of
                // magnitude, so the warps draw them from a queue (one shared-memory atomic per draw, the next draw in
                // flight while a unit runs), longest first: T | P | S | L | F, then the interior-loop cells in chunks of CH
                // (+7 % at 300 nt; in shared-memory configurations the static deal below is faster).
                constexpr int CH = 4;
                const int uP = nT, uS = uP + nP, uL = uS + nS, uF = uL + 2, uC = uF + nF;
                const int nc2 = (n2 + CH - 1) / CH, total = uC + nc2 + (n3 + CH - 1) / CH;
                int *head = &sm.wq[ph];
                if (tid == 0) sm.wq[ph ^ 1] = 0;
                auto draw = [&]() {
                    int v = 0;
                    if (lane == 0) v = atomicAdd(head, 1);
                    return __shfl_sync(full, v, 0);
                };
                int my = draw();
                while (my < total) {
                    const int nx = draw();
                    if (my < uP) {
                        unit_T(d0 + 1, my, ntile, ksh, kwsh);
                    } else if (my < uS) {
                        const int it = my - uP;
                        unit_P(it < nch2 ? d0 + 2 : d0 + 3, it < nch2 ? it : it - nch2);
                    } else if (my < uL) {
                        const int u = my - uS;
                        unit_S(u >= nseg0 ? d0 + 1 : d0, u >= nseg0 ? u - nseg0 : u);
                    } else if (my < uF) {
                        build_list(d0 + 4 + (my - uL));
                    } else if (my < uC) {
                        unit_F(d0 - 2, my - uF);
                    } else {
                        const int ci = my - uC, ds = ci >= nc2;
                        const int c = (ds ? ci - nc2 : ci) * CH;
                        unit_C(d0 + 2 + ds, c, min(c + CH, ds ? n3 : n2));
                    }
                    my = nx;
                }
            } else {
                const int uP = nS, uT = uP + nP, uF = uT + nT, uL = uF + nF, nH = uL + 2;
                for (int u = warp; u < nH; u += NW) {
                    if (u < uP) {
                        unit_S(u >= nseg0 ? d0 + 1 : d0, u >= nseg0 ? u - nseg0 : u);
                    } else if (u < uT) {
                        const int it = u - uP;
                        unit_P(it < nch2 ? d0 + 2 : d0 + 3, it < nch2 ? it : it - nch2);
                    } else if (u < uF) {
                        unit_T(d0 + 1, u - uT, ntile, ksh, kwsh);
                    } else if (u < uL) {
                        unit_F(d0 - 2, u - uF);
                    } else {
                        build_list(d0 + 4 + (u - uL));
                    }
                }
                // ---- C: interior loops of size >= 2 of the pairable cells of diagonals d0+2, d0+3 (rows <= d0-1): one
                // cell per pass, lane = loop size U with its seven taps (see the header).  The cells continue the round
                // robin of the units above.  (Same walk as unit_C; kept inline: as a lambda it costs 2.6 % at 120 nt.)  One byte
                // address per tap, the cell's scaled index added per load (+1 % at 120 nt, +2.4 % at 64 / 200 nt).
                int c = warp - nH % NW;
                if (c < 0) c += NW;
#pragma unroll 1
                for (int ds = 0; ds < 2; ds++) {
                    const int d = d0 + 2 + ds, n = ds ? n3 : n2;
                    if (c < n) {
                        const int slot = (d - 2 - UB) & (R32 - 1);
                        const unsigned sb = (unsigned)__cvta_generic_to_shared(smb);
                        const unsigned aA = sb + 2 * (kA + ((d - 2 - UA) & (R32 - 1)) * PR);
                        const unsigned aB10 = sb + 2 * (O_M8 + 10 + ((d - 2 - UB10) & (R32 - 1)) * PR);
                        const unsigned aB18 = sb + 2 * (O_M8 + 18 + ((d - 2 - UB18) & (R32 - 1)) * PR);
                        const unsigned aB26 = sb + 2 * (O_M8 + 26 + ((d - 2 - UB26) & (R32 - 1)) * PR);
                        const unsigned aC = sb + 2 * (kC + ((d - 2 - UC) & (R32 - 1)) * PR);
                        const unsigned aR = (unsigned)__cvta_generic_to_shared(sm.rpa + slot * PRW + 1);       // inner pair (i+1, j-1-U) and 1xn neighbour
                        const unsigned aL = (unsigned)__cvta_generic_to_shared(sm.rpq + slot * PRW + d - 1);   // inner pair (i+1+U, j-1) and 1xn neighbour
                        const unsigned aP = (unsigned)__cvta_generic_to_shared(sm.partc + (d & 3) * PR);
                        unsigned aLst = (unsigned)__cvta_generic_to_shared(reinterpret_cast<const int4 *>(sm.list) + (d & 3) * LP + c);
                        int4 en = lds_v4(aLst);
                        for (; c < n; c += NW) {
                            const int i = en.x, eI = en.y, e1 = en.z, eB = en.w;
                            aLst += NW * 16;
                            en = lds_v4(aLst);   // next entry (at most NW past the list end: still inside sm.list)
                            const unsigned i2 = 2 * i, i4 = 4 * i;
                            const unsigned wr = lds_u32(aR + i4), wl = lds_u32(aL + i4);
                            const int xa = lds_s16(aA + i2), xb10 = lds_s16(aB10 + i2), xb18 = lds_s16(aB18 + i2);
                            const int xb26 = lds_s16(aB26 + i2), xc = lds_s16(aC + i2);
                            const unsigned wm = __vmins2(wr, wl);
                            const int xb = (int)(short)(wm & 0xffffu), x1 = (int)wm >> 16;
                            int g = xa + cA;
                            g = __viaddmin_s32(xb10, cB10, g);
                            int g2 = xb18 + cB18;
                            g2 = __viaddmin_s32(xb26, cB26, g2);
                            g = __viaddmin_s32(xc, cC, g);
                            const int aB = xb + cSB, a1 = x1 + cS1;
                            int v = min(g, g2) + eI;
                            v = __viaddmin_s32(a1, e1, v);
                            v = __viaddmin_s32(aB, eB, v);
                            v = __reduce_min_sync(full, v);
                            if (lane == 0) sts_u16(aP + i2, v);   // <= INF16 + size and mismatch terms: fits
                        }
                    }
                    c -= n;
                }
            }
            __syncthreads();
        }

        // ---- exterior loop: stage C (+ stem term) back from the scratch row, then F5 sequentially (warp 0)
        {
            short *cx = sm.ne;
            const int ntri = tri4(W, W);
            for (int k = tid; k < ntri; k += NT) cx[k] = __ldcg(gC + k);
            for (int k = tid; k <= min(W, TURN + 1); k += NT) sm.f5[k] = 0;
            const int minw = __reduce_min_sync(full, minv);
            if (lane == 0) sm.minv[warp] = minw;
            __syncthreads();
            // F5[len] = min(F5[len-1], min_{i <= len-5} F5[i] + Cx(i, len-1)).  Eight consecutive lengths per round: every
            // term whose F5[i] is known when the round starts (i < len0) is a parallel minimum, one length per warp
            // (slices of the i range when there are more than eight warps, several lengths per warp when fewer); the
            // six terms that need F5 of the round itself (i = len0 .. len0+2 for the last three lengths) and the running
            // minimum along the block are folded in by one thread.
            constexpr int LPR = 8, NPART = NW > LPR ? NW / LPR : 1;
            for (int len0 = TURN + 2; len0 <= W; len0 += LPR) {
                for (int t = warp % LPR; t < LPR; t += NW) {
                    const int len = len0 + t, j = len - 1, part = warp / LPR;
                    int best = INF16;
                    if (len <= W && part < NPART)
                        for (int i = lane + 32 * part; i <= min(j - TURN - 1, len0 - 1); i += 32 * NPART)
                            best = min(best, sm.f5[i] + cx[tri4(j - i, W) + i]);
                    best = __reduce_min_sync(full, best);
                    if (lane == 0 && part < NPART) sm.fbest[t + LPR * part] = best;
                }
                __syncthreads();
                if (tid == 0) {
                    int f[LPR];
                    int run = sm.f5[len0 - 1];
#pragma unroll
                    for (int t = 0; t < LPR; t++) {
                        if (len0 + t <= W) {
#pragma unroll
                            for (int h = 0; h < NPART; h++) run = min(run, sm.fbest[t + LPR * h]);
                            // terms with i = len0 .. len - 5 (at most three): F5[i] was set earlier in this round
#pragma unroll
                            for (int q = 0; q + 5 <= t; q++) {
                                const int i = len0 + q, j = len0 + t - 1;
                                run = min(run, f[q] + cx[tri4(j - i, W) + i]);
                            }
                            f[t] = run;
                            sm.f5[len0 + t] = (short)run;
                        }
                    }
                }
                __syncthreads();
            }
            int mv = sm.minv[0];
            for (int q = 1; q < NW; q++) mv = min(mv, sm.minv[q]);
            if (tid == 0) L.e_out[fold] = mv < LOW16 ? MFE_REDO : (int)sm.f5[W];
            if (L.pair_tbl && mv >= LOW16) {   // native folds: structure (CTA-uniform branch)
                short *pt = sm.partc;
                if (warp == 0) {
                    const bool ok = traceback3<P, FMG>(sm, fm, T, cx, pt, W, lane);
                    if (!ok && lane == 0) L.e_out[fold] = MFE_REDO;   // the int32 kernel folds it again
                }
                __syncthreads();
                for (int k = tid; k < W; k += NT) L.pair_tbl[(size_t)fold * W + k] = pt[k];
            }
        }
    }
}

template <int P, int NW, int OCC, bool FMG = false>
void launch_mfe3_t(const MfeLaunch &L, const MfeTables *d_tab, int n_sm, cudaStream_t stream) {
    const size_t smem = sizeof(Smem3<P, FMG>);
    static bool cfg = false;
    if (!cfg) {
        cudaFuncSetAttribute(mfe3_kernel<P, NW, OCC, FMG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cfg = true;
    }
    const int grid = L.n_fold < n_sm * OCC ? L.n_fold : n_sm * OCC;
    mfe3_kernel<P, NW, OCC, FMG><<<grid, NW * 32, smem, stream>>>(L, d_tab, g_dtab3);
}

}  // namespace

static_assert(sizeof(Smem3<200>) <= 227 * 1024, "the 200-nt configuration must fit one SM");
static_assert(sizeof(Smem3<300, true>) <= 227 * 1024, "the 300-nt configuration must fit one SM");
static_assert(300 * 300 % 8 == 0, "the global matrix is cleared with 16-byte stores");
bool mfe3_supports(int W) { return g_mfe3_ok && W >= 16 && W <= 300; }

// scratch shorts per resident CTA: C (+ exterior stem term) by diagonal, and above 200 nt the FML matrix (300 x 300)
size_t mfe3_scratch_shorts_per_cta(int W) {
    const size_t tri = ((size_t)tri4(W, W) + 63) & ~(size_t)63;
    return tri + (W > 200 ? (size_t)300 * 300 : 0);
}

// scratch rows (one per resident CTA, the most any configuration launches)
int mfe3_max_ctas(int n_sm, int W) { return n_sm * (W <= 64 ? 4 : (W <= 120 ? 2 : 1)); }

void mfe3_upload_tables(const MfeTables &M) {
    static Tab3 h;
    // every entry below is stored as int16: a table value outside the envelope (INF entries of the stack / mismatch
    // tables included, which (short) would wrap) declines the table, and the int32 kernel folds instead
    bool fit = true;
    auto s16 = [&fit](int v) {
        fit = fit && v >= -TABLE_ENV16 && v <= TABLE_ENV16;
        return (short)v;
    };
    auto mm = [](int t, int a, int b) { return (t * 5 + a) * 5 + b; };
    static const int rt[8] = {0, 2, 1, 4, 3, 6, 5, 7};
    for (int a = 0; a < 8; a++)
        for (int b = 0; b < 8; b++) h.stack[a * 8 + b] = s16(M.stack[a][b]);
    for (int t = 0; t < 8; t++) {
        h.tAU[t] = s16(t > 2 ? M.TerminalAU : 0);
        h.rtype[t] = (unsigned char)rt[t];
        for (int a = 0; a < 5; a++)
            for (int b = 0; b < 5; b++) {
                h.mmI[mm(t, a, b)] = s16(M.mismatchI[t][a][b]);
                h.mm1n[mm(t, a, b)] = s16(M.mismatch1nI[t][a][b]);
                h.mm23[mm(t, a, b)] = s16(M.mismatch23I[t][a][b]);
                h.mmH[mm(t, a, b)] = s16(M.mismatchH[t][a][b]);
                h.mlclose[mm(t, a, b)] = s16(M.mismatchM[t][a][b] + (t > 2 ? M.TerminalAU : 0) + M.MLintern + M.MLclosing);
            }
        for (int a = 0; a < 6; a++)
            for (int b = 0; b < 6; b++) {
                int em = 0, ee = 0;
                if (a < 5 && b < 5) {
                    em = M.mismatchM[t][a][b];
                    ee = M.mismatchExt[t][a][b];
                } else if (a < 5) {
                    em = ee = M.dangle5[t][a];
                } else if (b < 5) {
                    em = ee = M.dangle3[t][b];
                }
                const int au = t > 2 ? M.TerminalAU : 0;
                h.mlstem[t * 36 + a * 6 + b] = s16(em + au + M.MLintern);
                h.ext[t * 36 + a * 6 + b] = s16(ee + au);
            }
    }
    for (int a = 0; a < 6; a++)
        for (int b = 0; b < 6; b++) h.ptype[a * 6 + b] = (unsigned char)((a < 5 && b < 5) ? pair_type(a, b) : 0);
    h.bulge1 = s16(M.bulge[1]);
    h.il5_ninio = s16(M.internal_loop[5] + M.ninio);
    h.MLbase = s16(M.MLbase);
    auto wk = [&](int k) { return s16(std::min(M.max_ninio, k * M.ninio)); };
    h.w1 = wk(1);
    h.w2 = wk(2);
    h.w3 = wk(3);
    h.w4 = wk(4);
    h.pad = 0;
    // the stencil / range-minimum split needs every asymmetry >= 5 to be capped and sane magnitudes
    g_mfe3_ok = fit && M.ninio >= 0 && 5 * M.ninio >= M.max_ninio && M.max_ninio >= 0 && M.max_ninio < 2000;
    static int sI[32], s1[32], sB[32], sC[32], s6[4];
    for (int u = 0; u < 32; u++) {
        const bool ok = u <= MAXLOOP && M.internal_loop[u < 31 ? u : 30] < INF;
        sI[u] = ok ? M.internal_loop[u] : INF16;
        sC[u] = ok ? M.internal_loop[u] + M.max_ninio : INF16;
        s1[u] = ok ? M.internal_loop[u] + std::min(M.max_ninio, (u - 2) * M.ninio) : INF16;
        sB[u] = (u <= MAXLOOP && M.bulge[u < 31 ? u : 30] < INF) ? M.bulge[u] : INF16;
    }
    for (int k = 0; k < 3; k++) {
        const int u1 = 2 + k, u2 = 6 - u1, diff = u1 > u2 ? u1 - u2 : u2 - u1;
        s6[k] = M.internal_loop[6] < INF ? M.internal_loop[6] + std::min(M.max_ninio, diff * M.ninio) : INF16;
    }
    s6[3] = INF16;
    cudaMemcpyToSymbol(c3_il, sI, sizeof(sI));
    cudaMemcpyToSymbol(c3_cap, sC, sizeof(sC));
    cudaMemcpyToSymbol(c3_size1, s1, sizeof(s1));
    cudaMemcpyToSymbol(c3_sizeB, sB, sizeof(sB));
    cudaMemcpyToSymbol(c3_sG6, s6, sizeof(s6));
    if (!g_dtab3) cudaMalloc(&g_dtab3, sizeof(Tab3));
    cudaMemcpy(g_dtab3, &h, sizeof(Tab3), cudaMemcpyHostToDevice);
}

void launch_mfe3(const MfeLaunch &L, const MfeTables *d_tab, int n_sm, cudaStream_t stream, int *n_launches) {
    if (L.n_fold <= 0) return;
    static const int nw = getenv("SFB_MFE3_WARPS") ? atoi(getenv("SFB_MFE3_WARPS")) : 12;  // tuning knob
    if (L.W <= 64)
        launch_mfe3_t<64, 4, 4>(L, d_tab, n_sm, stream);
    else if (L.W > 200)
        launch_mfe3_t<300, 16, 1, true>(L, d_tab, n_sm, stream);
    else if (L.W > 120)
        launch_mfe3_t<200, 16, 1>(L, d_tab, n_sm, stream);
    else if (nw == 4)
        launch_mfe3_t<120, 4, 2>(L, d_tab, n_sm, stream);
    else if (nw == 12)
        launch_mfe3_t<120, 12, 2>(L, d_tab, n_sm, stream);
    else if (nw == 16)
        launch_mfe3_t<120, 16, 2>(L, d_tab, n_sm, stream);
    else
        launch_mfe3_t<120, 8, 2>(L, d_tab, n_sm, stream);
    if (n_launches) (*n_launches)++;
}

}  // namespace sfb
