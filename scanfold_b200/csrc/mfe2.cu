// MFE fold kernel, second generation: a team of one or two warps per fold, energy only, windows up to 120 nt.
//
// Replaces the r background folds per window of energies()/rna_folder (ScanFoldFunctions.py:774-789,805-814)
// -- more than 99 % of all fold arithmetic of a scan.  The first-generation kernel (mfe.cu: one 256-thread CTA
// per fold, ~230 block barriers per fold, one fold resident per SM) is latency bound at 12 % warp occupancy;
// here a fold never leaves its warp, so there are no block barriers at all, and four folds are resident per SM.
//
// Layout per fold (shared memory, int16 dcal; INF16 = 16000, anything >= FIN16 = 4000 means "no structure"):
//   FML    folded diagonal-major rectangle, pitch P: diagonal dd <= W/2 sits in row dd, diagonal dd > W/2 in
//          the unused tail of row W - dd.  A split  FML[i,i+k] + FML[i+k+1,j]  then walks both operands with
//          compile-time strides (+P or -P+1), so a relaxation is 2 LDS + 1 VIADDMNMX and no address math.
//   RG/R1/RB  34-row rolling copies of C for the three separable interior-loop classes (generic, 1xn, bulge),
//          each already including the inner pair's mismatch / terminal-AU term.  A lane owns one pairable
//          cell (i,j) and runs over its <= 496 (u1,u2) candidates: LDS with an immediate offset + one
//          VIADDMNMX whose size term is a constant-bank operand.
//   RC/ctx 16-row rolling raw C and inner pair type for the nine table-driven loop shapes.
// C itself (plus its exterior-loop stem term) streams to an L2-resident scratch row per warp and is staged
// back once for the sequential F5 recurrence.
// Diagonals are processed two at a time (C of diagonals d and d+1 only depends on diagonals <= d-1), which
// keeps the 32 lanes busy with pairable cells.
// int16 storage is exact as long as no stored energy drops below LOW16; a fold that does is flagged and redone
// by the int32 kernel (mfe.cu) in the same stream, so results never depend on which kernel ran.
#include <cstdlib>

#include "device_common.cuh"

namespace sfb {
namespace {

constexpr int INF16 = 16000;
constexpr int TABLE_ENV16 = 2000;   // |table entry| the int16 arithmetic accepts (DESIGN §2)
constexpr int FIN16 = 4000;
constexpr int LOW16 = -12000;
constexpr int ROLL = 34;   // rows d-32 .. d+1 are live while a pair of diagonals (d, d+1) is computed
constexpr int RCR = 16;    // raw-C / type ring: rows d-7 .. d+1
constexpr int FOLDS_PER_CTA = 4;

struct alignas(16) Tab2 {
    short stack[64], mmI[200], mm1n[200], mm23[200], mmH[200];
    short mlclose[200];        // mismatchM + TerminalAU + MLintern + MLclosing (closing pair of a multiloop)
    short mlstem[8 * 36];      // [type][5' code][3' code], code 5 = no neighbour: E_MLstem
    short ext[8 * 36];         // E_ExtLoop likewise
    short tAU[8];
    short bulge1;              // bulge[1]
    short il5_ninio;           // internal_loop[5] + ninio   (2x3 loops)
    short MLbase;
    unsigned char ptype[36];   // pair type of codes a*6+b (code 5 = sentinel)
    unsigned char rtype[8];
};

__constant__ int c_sizeG[31][32];  // [u][u1]: internal_loop[u] + min(MAX_NINIO, |u1-u2|*ninio)
__constant__ int c_size1[32];      // 1xn loops of total size u
__constant__ int c_sizeB[32];      // bulge[u]
__constant__ int c_cap[32];        // internal_loop[u] + MAX_NINIO: every generic loop with |u1-u2| >= NEAR
Tab2 *g_dtab2 = nullptr;
bool g_mfe2_ok = false;            // the table set has the asymmetry cap structure the kernel assumes
constexpr int NEAR = 5;            // |u1-u2| >= NEAR  =>  the ninio term is capped (5*ninio >= MAX_NINIO, checked on upload)
constexpr unsigned INF16X2 = (unsigned)INF16 * 65537u;

template <int P>
struct FoldSmem {
    short roll[4 * ROLL * P];  // RG0 | RG1 (RG shifted by one element) | R1 | RB  (also the F5 staging area for C)
    short fml[(P / 2 + 1) * P];
    short rc[RCR * P];
    short dml[4 * P];
    short f5[P + 8];
    short list[2 * P];
    unsigned char ctx[RCR * P];
    unsigned char sx[P + 8];   // sx[k+1] = code of nucleotide k, sx[0] = sx[W+1] = 5
};

__host__ __device__ __forceinline__ int tri4(int d, int W) {  // first cell of diagonal d in the d >= 4 triangle
    return (d - 4) * W - ((d - 1) * d / 2 - 6);
}

// One u-block: candidates (u1, U-u1) of the separable classes of a cell whose inner diagonal is d-2-U.
//   rpG  the lane's view of the generic-class row: rpG[u1] is candidate u1 and &rpG[u1] is 4-byte aligned for
//        even u1 (lanes with odd i+1 read the copy that is shifted by one element), so two candidates come in
//        with one LDS.32;
//   rp1  &R1[row][i+1]; the bulge class sits ROLL*P further.
// Generic loops with |u1-u2| >= NEAR all carry the same size term c_cap[U], so they only need a running
// minimum (VIMNMX.S16x2 on packed pairs) and one add at the end of the block; the few near-symmetric ones,
// the two 1xn and the two bulge candidates take one VIADDMNMX each.
template <int U, int P>
__device__ __forceinline__ void ublock(const short *rpG, const short *rp1, int &g0, int &g1, int &a1, int &aB) {
    constexpr int OB = ROLL * P;
    if constexpr (U >= 2) {
        aB = __viaddmin_s32(rp1[OB], c_sizeB[U], aB);
        aB = __viaddmin_s32(rp1[OB + U], c_sizeB[U], aB);
    }
    if constexpr (U >= 4) {
        a1 = __viaddmin_s32(rp1[1], c_size1[U], a1);
        a1 = __viaddmin_s32(rp1[U - 1], c_size1[U], a1);
    }
    if constexpr (U >= 6) {
        unsigned f0 = INF16X2, f1 = INF16X2;
        int fs = INF16;
        bool anyfar = false;
#pragma unroll
        for (int k = 2; k <= U - 2; k += 2) {
            const int da = 2 * k - U, db = 2 * (k + 1) - U;
            const bool hasb = k + 1 <= U - 2;
            const bool fara = da >= NEAR || da <= -NEAR, farb = hasb && (db >= NEAR || db <= -NEAR);
            if (fara && farb) {
                const unsigned w = *reinterpret_cast<const unsigned *>(rpG + k);
                if ((k & 2) == 0) f0 = __vmins2(f0, w); else f1 = __vmins2(f1, w);
                anyfar = true;
            } else {
                if (fara) {
                    fs = min(fs, (int)rpG[k]);
                    anyfar = true;
                } else {
                    g0 = __viaddmin_s32(rpG[k], c_sizeG[U][k], g0);
                }
                if (hasb) {
                    if (farb) {
                        fs = min(fs, (int)rpG[k + 1]);
                        anyfar = true;
                    } else {
                        g1 = __viaddmin_s32(rpG[k + 1], c_sizeG[U][k + 1], g1);
                    }
                }
            }
        }
        if (anyfar) {
            const unsigned f = __vmins2(f0, f1);
            const int lo = (short)(f & 0xffffu), hi = (int)f >> 16;
            g0 = __viaddmin_s32(min(min(lo, hi), fs), c_cap[U], g0);
        }
    }
}

template <int U, int P>
struct UBlocks {
    __device__ __forceinline__ static void run(const short *roll, int goff, int loff, int &slot, int umax, int &g0,
                                               int &g1, int &a1, int &aB) {
        UBlocks<U - 1, P>::run(roll, goff, loff, slot, umax, g0, g1, a1, aB);
        if (U <= umax) {
            if constexpr (U >= 2) ublock<U, P>(roll + slot * P + goff, roll + slot * P + loff, g0, g1, a1, aB);
            slot = slot == 0 ? ROLL - 1 : slot - 1;
        }
    }
};
template <int P>
struct UBlocks<-1, P> {
    __device__ __forceinline__ static void run(const short *, int, int, int &, int, int &, int &, int &, int &) {}
};

__device__ int hairpin_special(const MfeTables *T, const Tab2 &tb, const unsigned char *sx, int i, int j, int type) {
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

// TW warps work on one fold ("team"); TW = 1 needs no block-level synchronisation at all, TW = 2 trades
// three 64-thread named barriers per diagonal pair for twice the resident warps per scheduler.
template <int TW>
__device__ __forceinline__ void team_sync(int team) {
    if constexpr (TW == 1)
        __syncwarp();
    else
        asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "n"(32 * TW) : "memory");
}

template <int P, int TW>
__global__ void __launch_bounds__(FOLDS_PER_CTA * 32 * TW, 1)
mfe2_kernel(MfeLaunch L, const MfeTables *__restrict__ T, const Tab2 *__restrict__ gtab) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Tab2 &tb = *reinterpret_cast<Tab2 *>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int team = warp / TW, tw = warp % TW, tlane = tw * 32 + lane;
    constexpr int TL = 32 * TW;
    FoldSmem<P> &sm = *reinterpret_cast<FoldSmem<P> *>(smem_raw + ((sizeof(Tab2) + 15) & ~15) +
                                                       (size_t)team * ((sizeof(FoldSmem<P>) + 15) & ~15));
    {
        const int *src = reinterpret_cast<const int *>(gtab);
        int *dst = reinterpret_cast<int *>(&tb);
        static_assert(sizeof(Tab2) % 4 == 0, "Tab2 is copied as 32-bit words");
        for (int k = threadIdx.x; k < (int)(sizeof(Tab2) / 4); k += blockDim.x) dst[k] = src[k];
    }
    __syncthreads();

    const int W = L.W, H = W / 2;
    const unsigned full = 0xffffffffu;
    short *gC = reinterpret_cast<short *>(L.gscratch) + (size_t)(blockIdx.x * FOLDS_PER_CTA + team) * L.gscratch_per_cta;
    short *RG = sm.roll;
    const unsigned char *sx = sm.sx;
    short *list = sm.list + tw * P;

    for (int fold = blockIdx.x * FOLDS_PER_CTA + team; fold < L.n_fold; fold += gridDim.x * FOLDS_PER_CTA) {
        // ---- prologue: sequence with sentinels, INF in every rolling row
        for (int k = tlane; k < W + 2; k += TL)
            sm.sx[k] = (k == 0 || k == W + 1) ? 5 : L.seqs[(size_t)fold * W + k - 1];
        {
            const int4 inf4 = make_int4(INF16 * 65537, INF16 * 65537, INF16 * 65537, INF16 * 65537);
            int4 *p = reinterpret_cast<int4 *>(sm.roll);
            for (int k = tlane; k < (int)(sizeof(sm.roll) / 16); k += TL) p[k] = inf4;
            p = reinterpret_cast<int4 *>(sm.rc);
            for (int k = tlane; k < (int)(sizeof(sm.rc) / 16); k += TL) p[k] = inf4;
            p = reinterpret_cast<int4 *>(sm.dml);
            for (int k = tlane; k < (int)(sizeof(sm.dml) / 16); k += TL) p[k] = inf4;
        }
        int minv = 0;
        team_sync<TW>(team);

        for (int d0 = TURN + 1; d0 < W; d0 += 2) {
            const int nd = d0 + 1 < W ? 2 : 1;
            // ---- phase T: pair types, compaction of the pairable cells (TW = 2: one diagonal per warp)
            int nlist = 0;
            for (int ds = tw; ds < nd; ds += TW) {
                const int d = d0 + ds, ncells = W - d, slot = d % ROLL, t4 = tri4(d, W);
                for (int i0 = 0; i0 < ncells; i0 += 32) {
                    const int i = i0 + lane;
                    int t = 0;
                    if (i < ncells) {
                        t = tb.ptype[sx[i + 1] * 6 + sx[i + d + 1]];
                        sm.ctx[(d & (RCR - 1)) * P + i] = tb.rtype[t];
                        if (!t) {
                            sm.rc[(d & (RCR - 1)) * P + i] = INF16;
                            RG[slot * P + i] = INF16;
                            RG[(ROLL + slot) * P + i + 1] = INF16;
                            RG[(2 * ROLL + slot) * P + i] = INF16;
                            RG[(3 * ROLL + slot) * P + i] = INF16;
                            gC[t4 + i] = INF16;
                        }
                    }
                    const unsigned m = __ballot_sync(full, t != 0);
                    if (t) list[nlist + __popc(m & ((1u << lane) - 1))] = (short)(i | (ds << 8));
                    nlist += __popc(m);
                }
            }
            __syncwarp();
            // ---- phase C: one lane per pairable cell
            const int dhi = TW == 1 ? d0 + nd - 1 : d0 + tw;
            const int umax = min(MAXLOOP, dhi - 2 - (TURN + 1));
            const int hp0 = T->hairpin_len[d0 - 1], hp1 = T->hairpin_len[d0];
            for (int base = 0; base < nlist; base += 32) {
                const bool active = base + lane < nlist;
                const int code = active ? list[base + lane] : (TW == 1 ? 0 : tw << 8);
                const int i = code & 0xff, ds = code >> 8, d = d0 + ds, j = i + d;
                const int type = tb.ptype[sx[i + 1] * 6 + sx[j + 1]];
                const int si1 = sx[i + 2], sj1 = sx[j];
                const int mi = (type * 5 + si1) * 5 + sj1;
                int g0 = INF16, g1 = INF16, a1 = INF16, aB = INF16, aT = INF16;
                // the nine table-driven shapes
                {
                    auto inner = [&](int u1, int u2, int &c, int &t2, int &sp1, int &sq1) {
                        const int dd = d - 2 - u1 - u2, p = i + 1 + u1, q = j - 1 - u2;
                        const bool ok = dd > TURN;
                        c = ok ? sm.rc[(dd & (RCR - 1)) * P + p] : INF16;
                        t2 = ok ? sm.ctx[(dd & (RCR - 1)) * P + p] : 0;
                        sp1 = sx[p];       // S[p-1]
                        sq1 = sx[q + 2];   // S[q+1]
                    };
                    int c, t2, sp1, sq1;
                    inner(0, 0, c, t2, sp1, sq1);
                    aT = min(aT, c + tb.stack[type * 8 + t2]);
                    inner(0, 1, c, t2, sp1, sq1);
                    aT = min(aT, c + tb.bulge1 + tb.stack[type * 8 + t2]);
                    inner(1, 0, c, t2, sp1, sq1);
                    aT = min(aT, c + tb.bulge1 + tb.stack[type * 8 + t2]);
                    inner(1, 1, c, t2, sp1, sq1);
                    aT = min(aT, c + __ldg(&T->int11[type][t2][si1][sj1]));
                    inner(1, 2, c, t2, sp1, sq1);
                    aT = min(aT, c + __ldg(&T->int21[type][t2][si1][sq1][sj1]));
                    inner(2, 1, c, t2, sp1, sq1);
                    aT = min(aT, c + __ldg(&T->int21[t2][type][sq1][si1][sp1]));
                    inner(2, 2, c, t2, sp1, sq1);
                    aT = min(aT, c + __ldg(&T->int22[type][t2][si1][sp1][sq1][sj1]));
                    inner(2, 3, c, t2, sp1, sq1);
                    aT = min(aT, c + tb.il5_ninio + tb.mm23[mi] + tb.mm23[(t2 * 5 + sq1) * 5 + sp1]);
                    inner(3, 2, c, t2, sp1, sq1);
                    aT = min(aT, c + tb.il5_ninio + tb.mm23[mi] + tb.mm23[(t2 * 5 + sq1) * 5 + sp1]);
                }
                // separable classes
                {
                    int slot = (d - 2) % ROLL;
                    const int par = (i + 1) & 1;
                    UBlocks<MAXLOOP, P>::run(RG, (par ? ROLL * P : 0) + i + 1 + par, 2 * ROLL * P + i + 1, slot, umax, g0, g1,
                                             a1, aB);
                }
                int e = min(g0, g1) + tb.mmI[mi];
                e = min(e, a1 + tb.mm1n[mi]);
                e = min(e, aB + tb.tAU[type]);
                e = min(e, aT);
                int eh = (ds ? hp1 : hp0) + tb.mmH[mi];
                if (d <= 7 && active) eh = hairpin_special(T, tb, sx, i, j, type);
                e = min(e, eh);
                {
                    const int dm = sm.dml[((d - 2) & 3) * P + i + 1];
                    e = min(e, dm + tb.mlclose[(tb.rtype[type] * 5 + sj1) * 5 + si1]);
                }
                if (active) {
                    if (e >= FIN16) e = INF16;
                    minv = min(minv, e);
                    const int slot = d % ROLL;
                    sm.rc[(d & (RCR - 1)) * P + i] = (short)e;
                    int vg = INF16, v1 = INF16, vb = INF16;
                    if (i > 0 && j < W - 1 && e < FIN16) {
                        const int t2 = tb.rtype[type];
                        const int m2 = (t2 * 5 + sx[j + 2]) * 5 + sx[i];
                        vg = e + tb.mmI[m2];
                        v1 = e + tb.mm1n[m2];
                        vb = e + tb.tAU[t2];
                    }
                    RG[slot * P + i] = (short)vg;
                    RG[(ROLL + slot) * P + i + 1] = (short)vg;
                    RG[(2 * ROLL + slot) * P + i] = (short)v1;
                    RG[(3 * ROLL + slot) * P + i] = (short)vb;
                    gC[tri4(d, W) + i] = (short)(e < FIN16 ? e + tb.ext[type * 36 + sx[i] * 6 + sx[j + 2]] : INF16);
                }
            }
            team_sync<TW>(team);
            // ---- phase M: FML of diagonal d0, then d0 + 1
            for (int ds = 0; ds < nd; ds++) {
                const int d = d0 + ds, ncells = W - d;
                const int klo = TURN + 1, khi = d - 2 - TURN;       // split k: FML[i,i+k] + FML[i+k+1,j]
                const int kb = d - 1 - H;                            // operand B is in the low half for k >= kb
                for (int i0 = tw * 32; i0 < ncells; i0 += TL) {
                    const int i = min(i0 + lane, ncells - 1);
                    int m0 = 2 * INF16, m1 = 2 * INF16, m2 = 2 * INF16, m3 = 2 * INF16;
                    int k = klo;
                    {   // segment 1: A low (+P), B high (+P)
                        const int kend = min(kb - 1, khi);
                        const short *pa = sm.fml + k * P + i;
                        const short *pb = sm.fml + (W - d + 1 + k) * P + d + i;
                        for (; k + 3 <= kend; k += 4, pa += 4 * P, pb += 4 * P) {
                            m0 = __viaddmin_s32(pa[0], pb[0], m0);
                            m1 = __viaddmin_s32(pa[P], pb[P], m1);
                            m2 = __viaddmin_s32(pa[2 * P], pb[2 * P], m2);
                            m3 = __viaddmin_s32(pa[3 * P], pb[3 * P], m3);
                        }
                        for (; k <= kend; k++, pa += P, pb += P) m0 = __viaddmin_s32(pa[0], pb[0], m0);
                    }
                    {   // segment 2: A low (+P), B low (-P+1)
                        const int kend = min(H, khi);
                        const short *pa = sm.fml + k * P + i;
                        const short *pb = sm.fml + (d - 1 - k) * P + i + k + 1;
                        for (; k + 7 <= kend; k += 8, pa += 8 * P, pb -= 8 * (P - 1)) {
                            m0 = __viaddmin_s32(pa[0], pb[0], m0);
                            m1 = __viaddmin_s32(pa[P], pb[-(P - 1)], m1);
                            m2 = __viaddmin_s32(pa[2 * P], pb[-2 * (P - 1)], m2);
                            m3 = __viaddmin_s32(pa[3 * P], pb[-3 * (P - 1)], m3);
                            m0 = __viaddmin_s32(pa[4 * P], pb[-4 * (P - 1)], m0);
                            m1 = __viaddmin_s32(pa[5 * P], pb[-5 * (P - 1)], m1);
                            m2 = __viaddmin_s32(pa[6 * P], pb[-6 * (P - 1)], m2);
                            m3 = __viaddmin_s32(pa[7 * P], pb[-7 * (P - 1)], m3);
                        }
                        for (; k <= kend; k++, pa += P, pb -= P - 1) m0 = __viaddmin_s32(pa[0], pb[0], m0);
                    }
                    {   // segment 3: A high (-P+1), B low (-P+1)
                        const short *pa = sm.fml + (W - k) * P + k + i;
                        const short *pb = sm.fml + (d - 1 - k) * P + i + k + 1;
                        for (; k + 3 <= khi; k += 4, pa -= 4 * (P - 1), pb -= 4 * (P - 1)) {
                            m0 = __viaddmin_s32(pa[0], pb[0], m0);
                            m1 = __viaddmin_s32(pa[-(P - 1)], pb[-(P - 1)], m1);
                            m2 = __viaddmin_s32(pa[-2 * (P - 1)], pb[-2 * (P - 1)], m2);
                            m3 = __viaddmin_s32(pa[-3 * (P - 1)], pb[-3 * (P - 1)], m3);
                        }
                        for (; k <= khi; k++, pa -= P - 1, pb -= P - 1) m0 = __viaddmin_s32(pa[0], pb[0], m0);
                    }
                    int dec = min(min(m0, m1), min(m2, m3));
                    if (dec >= FIN16) dec = INF16;
                    int m = dec;
                    if (d - 1 > TURN) {
                        const short *prev = sm.fml + (d - 1 <= H ? (d - 1) * P + i : (W - d + 1) * P + d - 1 + i);
                        m = min(m, min(prev[0], prev[1]) + tb.MLbase);
                    }
                    const int c = sm.rc[(d & (RCR - 1)) * P + i];
                    const int type = tb.rtype[sm.ctx[(d & (RCR - 1)) * P + i]];
                    m = min(m, c + tb.mlstem[type * 36 + sx[i] * 6 + sx[i + d + 2]]);
                    if (m >= FIN16) m = INF16;
                    if (i0 + lane < ncells) {
                        minv = min(minv, m);
                        sm.dml[(d & 3) * P + i] = (short)dec;
                        sm.fml[d <= H ? d * P + i : (W - d) * P + d + i] = (short)m;
                    }
                }
                team_sync<TW>(team);
            }
        }

        // ---- exterior loop: stage C (+ stem term) back from the scratch row, then F5 sequentially (warp 0)
        {
            short *cx = sm.roll;
            const int ntri = tri4(W, W);
            for (int k = tlane; k < ntri; k += TL) cx[k] = __ldcg(gC + k);
            for (int k = tlane; k <= min(W, TURN + 1); k += TL) sm.f5[k] = 0;
            minv = __reduce_min_sync(full, minv);
            if (lane == 0) sm.f5[P + 2 + tw] = (short)max(minv, -32000);
            team_sync<TW>(team);
            if (tw == 0) {
                for (int len = TURN + 2; len <= W; len++) {
                    const int j = len - 1;
                    int best = INF16;
                    for (int i = lane; i <= j - TURN - 1; i += 32) best = min(best, sm.f5[i] + cx[tri4(j - i, W) + i]);
                    best = __reduce_min_sync(full, best);
                    if (lane == 0) sm.f5[len] = (short)min((int)sm.f5[len - 1], best);
                    __syncwarp();
                }
                if (lane == 0) {
                    int mv = sm.f5[P + 2];
                    for (int q = 1; q < TW; q++) mv = min(mv, (int)sm.f5[P + 2 + q]);
                    L.e_out[fold] = mv < LOW16 ? MFE_REDO : (int)sm.f5[W];
                }
            }
        }
        team_sync<TW>(team);
    }
}

}  // namespace

size_t mfe2_scratch_shorts_per_warp(int W) { return ((size_t)tri4(W, W) + 63) & ~(size_t)63; }

bool mfe2_supports(int W) { return g_mfe2_ok && W >= 16 && W <= 120; }

int mfe2_grid_size(int n_sm, int n_fold) {
    const int need = (n_fold + FOLDS_PER_CTA - 1) / FOLDS_PER_CTA;
    return need < n_sm ? need : n_sm;
}

void mfe2_upload_tables(const MfeTables &M) {
    static Tab2 h;
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
    static int sG[31][32], s1[32], sB[32], sC[32];
    g_mfe2_ok = fit && M.ninio >= 0 && NEAR * M.ninio >= M.max_ninio;
    for (int u = 0; u <= MAXLOOP; u++) {
        sC[u] = M.internal_loop[u] < INF ? M.internal_loop[u] + M.max_ninio : INF16;
        sB[u] = M.bulge[u] < INF ? M.bulge[u] : INF16;
        s1[u] = M.internal_loop[u] < INF ? M.internal_loop[u] + std::min(M.max_ninio, (u - 2) * M.ninio) : INF16;
        for (int u1 = 0; u1 < 32; u1++) {
            const int u2 = u - u1, diff = u1 > u2 ? u1 - u2 : u2 - u1;
            sG[u][u1] = (u1 <= u && M.internal_loop[u] < INF) ? M.internal_loop[u] + std::min(M.max_ninio, diff * M.ninio) : INF16;
        }
    }
    cudaMemcpyToSymbol(c_sizeG, sG, sizeof(sG));
    cudaMemcpyToSymbol(c_size1, s1, sizeof(s1));
    cudaMemcpyToSymbol(c_sizeB, sB, sizeof(sB));
    cudaMemcpyToSymbol(c_cap, sC, sizeof(sC));
    if (!g_dtab2) cudaMalloc(&g_dtab2, sizeof(Tab2));
    cudaMemcpy(g_dtab2, &h, sizeof(Tab2), cudaMemcpyHostToDevice);
}

template <int P, int TW>
static void launch_mfe2_t(const MfeLaunch &L, const MfeTables *d_tab, int grid, cudaStream_t stream) {
    const size_t smem = ((sizeof(Tab2) + 15) & ~15) + FOLDS_PER_CTA * ((sizeof(FoldSmem<P>) + 15) & ~15);
    static bool cfg = false;
    if (!cfg) {
        cudaFuncSetAttribute(mfe2_kernel<P, TW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cfg = true;
    }
    mfe2_kernel<P, TW><<<grid, FOLDS_PER_CTA * 32 * TW, smem, stream>>>(L, d_tab, g_dtab2);
}

void launch_mfe2(const MfeLaunch &L, const MfeTables *d_tab, int n_sm, cudaStream_t stream, int *n_launches) {
    if (L.n_fold <= 0) return;
    const int grid = mfe2_grid_size(n_sm, L.n_fold);
    static const int tw = getenv("SFB_MFE2_TEAM") ? atoi(getenv("SFB_MFE2_TEAM")) : 2;  // warps per fold (tuning knob)
    if (L.W <= 64) {
        if (tw == 1) launch_mfe2_t<64, 1>(L, d_tab, grid, stream);
        else launch_mfe2_t<64, 2>(L, d_tab, grid, stream);
    } else {
        if (tw == 1) launch_mfe2_t<120, 1>(L, d_tab, grid, stream);
        else launch_mfe2_t<120, 2>(L, d_tab, grid, stream);
    }
    if (n_launches) (*n_launches)++;
}

}  // namespace sfb
