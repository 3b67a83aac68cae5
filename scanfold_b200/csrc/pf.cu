// Partition function (McCaskill inside/outside, scaled fp64), base-pair probabilities, ensemble
// diversity and centroid for sm_100a.
//
// Replaces fc.pf(), fc.centroid(), fc.mean_bp_distance() -- ScanFold.py:498,503-504 / :514,518-519 /
// :525-527.  One CTA per window (persistent grid).  Both passes are anti-diagonal wavefronts over
// diagonal-major triangular matrices: inside fills qb/qm/qm1 for growing d = j - i, outside fills the
// pair "outside" weights P for shrinking d using two auxiliary matrices X1/X2 (right part of the
// enclosing multiloop with / without further stems) so that every cell is an O(W) sum.  The ED sum and
// the centroid threshold are fused into the last sweep; bpp is only written out on request.
#include "device_common.cuh"

namespace sfb {
namespace {

constexpr int NT = 256;
constexpr int NCAND = 496;

struct PfSmall {
    double expstack[64];
    double mmI[200], mm1n[200], mm23[200], mmM[200], mmExt[200], mmH[200];
    double d5[40], d3[40];
    double bulge[31], il[31], ninio[31];
    double expMLbase, expMLclosing, expMLintern, expTermAU, kT, pf_scale;
    short cand[NCAND];  // u1 | u2 << 5 | class << 10
    int ncand_upto[32];
    double fac[NCAND];  // separable classes: size factor * scale[u+2] of candidate ci (0 for table-driven shapes)
    int rowoff[32];     // ring row of the inner (inside) / outer (outside) diagonal for total loop size u
};

// Interior loops whose Boltzmann factor separates into (size term) x (outer mismatch) x (inner mismatch):
// the inner-pair part is folded into 34-row ring copies of qb (inside) / P (outside) when that cell is final,
// so a candidate costs one load and one FMA instead of a full loop-energy evaluation.
enum { PCLS_GENERIC = 0, PCLS_1N = 1, PCLS_BULGE = 2, PCLS_TABLE = 3 };
constexpr int PRING = 34;

struct PfCtx {
    const PfTables *T;
    const MfeTables *M;  // special-loop keys
    const PfSmall *s;
    const uint8_t *S;
    const int32_t *sc;
    const double *scale;
    int W;
    HcCtx h;
};

__device__ __forceinline__ int mm_idx(int t, int a, int b) { return (t * 5 + a) * 5 + b; }

__device__ double x_hairpin(const PfCtx &c, int i, int j, int type) {
    int u = j - i - 1;
    double z = c.T->exphairpin_len[u];
    if (u < 3) return z;
    if (u == 4) {
        int key = loop_key_dev(c.S, i, 6);
        for (int k = 0; k < c.M->n_tetra; k++)
            if (c.M->tetra_key[k] == key) return c.T->exptetra[k];
    } else if (u == 6) {
        int key = loop_key_dev(c.S, i, 8);
        for (int k = 0; k < c.M->n_hexa; k++)
            if (c.M->hexa_key[k] == key) return c.T->exphexa[k];
    } else if (u == 3) {
        int key = loop_key_dev(c.S, i, 5);
        for (int k = 0; k < c.M->n_tri; k++)
            if (c.M->tri_key[k] == key) return c.T->exptri[k];
        return type > 2 ? z * c.s->expTermAU : z;
    }
    return z * c.s->mmH[mm_idx(type, c.S[i + 1], c.S[j - 1])];
}

__device__ double x_intloop(const PfCtx &c, int u1, int u2, int type, int t2, int si1, int sj1, int sp1, int sq1) {
    const PfSmall &s = *c.s;
    int ul = max(u1, u2), us = min(u1, u2);
    if (ul == 0) return s.expstack[type * 8 + t2];
    if (us == 0) {
        double z = s.bulge[ul];
        if (ul == 1)
            z *= s.expstack[type * 8 + t2];
        else {
            if (type > 2) z *= s.expTermAU;
            if (t2 > 2) z *= s.expTermAU;
        }
        return z;
    }
    if (us == 1) {
        if (ul == 1) return c.T->expint11[type][t2][si1][sj1];
        if (ul == 2) {
            if (u1 == 1) return c.T->expint21[type][t2][si1][sq1][sj1];
            return c.T->expint21[t2][type][sq1][si1][sp1];
        }
        return s.il[ul + us] * s.mm1n[mm_idx(type, si1, sj1)] * s.mm1n[mm_idx(t2, sq1, sp1)] * s.ninio[ul - us];
    }
    if (us == 2) {
        if (ul == 2) return c.T->expint22[type][t2][si1][sp1][sq1][sj1];
        if (ul == 3) return s.il[5] * s.mm23[mm_idx(type, si1, sj1)] * s.mm23[mm_idx(t2, sq1, sp1)] * s.ninio[1];
    }
    return s.il[ul + us] * s.mmI[mm_idx(type, si1, sj1)] * s.mmI[mm_idx(t2, sq1, sp1)] * s.ninio[ul - us];
}

__device__ __forceinline__ double x_mlstem(const PfSmall &s, int type, int si1, int sj1) {
    double z = 1.;
    if (si1 >= 0 && sj1 >= 0)
        z = s.mmM[mm_idx(type, si1, sj1)];
    else if (si1 >= 0)
        z = s.d5[type * 5 + si1];
    else if (sj1 >= 0)
        z = s.d3[type * 5 + sj1];
    if (type > 2) z *= s.expTermAU;
    return z * s.expMLintern;
}

__device__ __forceinline__ double x_extloop(const PfSmall &s, int type, int si1, int sj1) {
    double z = 1.;
    if (si1 >= 0 && sj1 >= 0)
        z = s.mmExt[mm_idx(type, si1, sj1)];
    else if (si1 >= 0)
        z = s.d5[type * 5 + si1];
    else if (sj1 >= 0)
        z = s.d3[type * 5 + sj1];
    if (type > 2) z *= s.expTermAU;
    return z;
}

__device__ __forceinline__ double x_sc_stack(const PfCtx &c, int i, int j, int p, int q) {
    if (!c.sc) return 1.;
    int e = c.sc[i + 1] + c.sc[p + 1] + c.sc[q + 1] + c.sc[j + 1];
    return exp(-(double)e * 10. / c.s->kT);
}

__device__ __forceinline__ int floor_pow2(int x) { return x <= 1 ? 1 : 1 << (31 - __clz(x)); }

__device__ __forceinline__ double group_sum(double v, int G) {
    for (int o = 1; o < G; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

#ifndef SFB_PF_MINB
#define SFB_PF_MINB 6   // resident CTAs per SM: measured 3 -> 9.99 k, 4 -> 10.6 k, 6 -> 13.0 k, 8 -> 8.9 k windows/s at 200 nt
#endif
// PAIRPROB: the launch carries a pair-probability table; a fold whose dG and ED are finite commits p = P * qb of every cell
// (both triangles are still in the CTA's scratch at its end)
template <bool PAIRPROB>
__global__ void __launch_bounds__(NT, SFB_PF_MINB) pf_kernel(PfLaunch L, const MfeTables *__restrict__ MT,
                                                const PfTables *__restrict__ T, PairProbCommit pp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int W = L.W;
    const int tid = threadIdx.x, lane = tid & 31;
    const size_t ntri = (size_t)W * (W + 1) / 2;

    PfSmall *st = reinterpret_cast<PfSmall *>(smem_raw);
    double *dp = reinterpret_cast<double *>(smem_raw + ((sizeof(PfSmall) + 15) & ~15));
    const int nscale = max(W, MAXLOOP) + 4;   // st->fac reads scale[u1 + u2 + 2] up to MAXLOOP + 2 at every W
    double *scale = dp;   dp += nscale;
    double *eMLb = dp;    dp += W + 4;
    double *q5 = dp;      dp += W + 2;
    double *q3 = dp;      dp += W + 2;
    double *red = dp;     dp += 8;
    int *ip = reinterpret_cast<int *>(dp);
    int *scs = ip;        ip += W + 2;
    int *misc = ip;       ip += 4;
    int *bstk = ip;       ip += W + 2;
    int16_t *list = reinterpret_cast<int16_t *>(ip);
    int16_t *mate = list + W;
    int16_t *cen = mate + W;
    uint8_t *S = reinterpret_cast<uint8_t *>(cen + W);
    uint8_t *hcf = S + W + 4;
    uint8_t *ctype = hcf + W + 4;

    // qb and P stay diagonal-major triangles (read along diagonals); every matrix an O(W) sum walks lives in the
    // orientation that makes the walk contiguous, so the lanes that share a cell read one row segment per load:
    //   qmR [i][k] row-major, qmC [k][i] column-major (both written per cell), qm1C column-major,
    //   X1C / X2C column-major, PMR row-major.  Entries with j - i <= TURN are never read.
    const size_t sq = (size_t)W * W;
    double *g = L.gscratch + (long long)blockIdx.x * L.gscratch_per_cta;
    double *qb = g;            g += ntri;
    double *Pm = g;            g += ntri;
    double *qmR = g;           g += sq;
    double *qmC = g;           g += sq;
    double *qm1C = g;          g += sq;
    double *PMR = g;           g += sq;
    double *X1C = g;           g += sq;
    double *X2C = g;           g += sq;
    double *ring = g;          // [3][PRING][W]: generic | 1xn | bulge class copies
#define RM(i, j) ((size_t)(i) * W + (j))
#define CM(i, j) ((size_t)(j) * W + (i))

    {
        auto cp = [&](double *dst, const double *s, int n) {
            for (int k = tid; k < n; k += NT) dst[k] = s[k];
        };
        cp(st->expstack, &T->expstack[0][0], 64);
        cp(st->mmI, &T->expmismatchI[0][0][0], 200);
        cp(st->mm1n, &T->expmismatch1nI[0][0][0], 200);
        cp(st->mm23, &T->expmismatch23I[0][0][0], 200);
        cp(st->mmM, &T->expmismatchM[0][0][0], 200);
        cp(st->mmExt, &T->expmismatchExt[0][0][0], 200);
        cp(st->mmH, &T->expmismatchH[0][0][0], 200);
        cp(st->d5, &T->expdangle5[0][0], 40);
        cp(st->d3, &T->expdangle3[0][0], 40);
        cp(st->bulge, T->expbulge, 31);
        cp(st->il, T->expinternal, 31);
        cp(st->ninio, T->expninio, 31);
        if (tid == 0) {
            st->expMLbase = T->expMLbase;
            st->expMLclosing = T->expMLclosing;
            st->expMLintern = T->expMLintern;
            st->expTermAU = T->expTermAU;
            st->kT = T->kT;
            st->pf_scale = L.pf_scale > 0. ? L.pf_scale : T->pf_scale;
            int n = 0;
            for (int u = 0; u <= MAXLOOP; u++) {
                for (int u1 = 0; u1 <= u; u1++) {
                    const int u2 = u - u1, ul = max(u1, u2), us = min(u1, u2);
                    int cls = PCLS_TABLE;
                    if (us == 0 && ul >= 2) cls = PCLS_BULGE;
                    else if (us == 1 && ul >= 3) cls = PCLS_1N;
                    else if (us >= 2 && !(us == 2 && ul <= 3)) cls = PCLS_GENERIC;
                    st->cand[n++] = (short)(u1 | (u2 << 5) | (cls << 10));
                }
                st->ncand_upto[u] = n;
            }
            scale[0] = 1.;
            eMLb[0] = 1.;
            for (int k = 1; k < nscale; k++) scale[k] = scale[k - 1] / st->pf_scale;
            for (int k = 1; k < W + 4; k++) eMLb[k] = eMLb[k - 1] * T->expMLbase / st->pf_scale;
        }
    }
    __syncthreads();
    for (int ci = tid; ci < NCAND; ci += NT) {
        const int cd = st->cand[ci], u1 = cd & 31, u2 = (cd >> 5) & 31, cls = cd >> 10;
        const int ul = max(u1, u2), us = min(u1, u2);
        double f = 0.;
        if (cls == PCLS_BULGE) f = st->bulge[ul];
        else if (cls == PCLS_1N || cls == PCLS_GENERIC) f = st->il[ul + us] * st->ninio[ul - us];
        st->fac[ci] = f * scale[u1 + u2 + 2];
    }
    __syncthreads();

    PfCtx c;
    c.T = T;
    c.M = MT;
    c.s = st;
    c.S = S;
    c.scale = scale;
    c.W = W;
    c.h.S = S;
    c.h.W = W;
    c.h.max_span = L.max_span;
    const double closing = st->expMLclosing;

#define TRI(d, i) (tri_off((d), W) + (i))

    for (int fold = blockIdx.x; fold < L.n_fold; fold += gridDim.x) {
        for (int k = tid; k < W; k += NT) {
            S[k] = L.seqs[(long long)fold * W + k];
            cen[k] = 0;
        }
        c.h.hcf = nullptr;
        c.h.mate = nullptr;
        c.h.n_enf = 0;
        c.sc = nullptr;
        if (L.hc) {
            for (int k = tid; k < W; k += NT) {
                char ch = (char)L.hc[(long long)fold * W + k];
                hcf[k] = (ch == 'x' ? 1 : 0) | (ch == '<' ? 2 : 0) | (ch == '>' ? 4 : 0);
                mate[k] = -1;
            }
            c.h.hcf = hcf;
            c.h.mate = mate;
        }
        if (L.sc) {
            for (int k = tid; k <= W; k += NT) scs[k] = L.sc[(long long)fold * (W + 1) + k];
            c.sc = scs;
        }
        __syncthreads();
        if (L.hc && tid == 0) {
            int sp = 0, n_enf = 0;
            for (int k = 0; k < W; k++) {
                char ch = (char)L.hc[(long long)fold * W + k];
                if (ch == '(')
                    bstk[sp++] = k;
                else if (ch == ')' && sp > 0) {
                    int a = bstk[--sp];
                    mate[a] = (int16_t)k;
                    mate[k] = (int16_t)a;
                    n_enf++;
                }
            }
            misc[1] = n_enf;
        }
        __syncthreads();
        if (L.hc) c.h.n_enf = misc[1];

        // ================= inside =================
        for (int d = TURN + 1; d < W; d++) {
            const int ncells = W - d;
            const int tri_d = tri_off(d, W);
            if (tid == 0) misc[0] = 0;
            if (tid < 32) st->rowoff[tid] = ((d - 2 - tid + 2 * PRING) % PRING) * W;
            __syncthreads();
            const int ring_row = (d % PRING) * W;
            for (int i = tid; i < ncells; i += NT) {
                int t = allowed_type(c.h, i, i + d);
                ctype[i] = (uint8_t)t;
                if (!t) {
                    qb[tri_d + i] = 0.;
                    ring[ring_row + i] = 0.;
                    ring[PRING * W + ring_row + i] = 0.;
                    ring[2 * PRING * W + ring_row + i] = 0.;
                } else
                    list[atomicAdd(&misc[0], 1)] = (int16_t)i;
            }
            __syncthreads();
            {   // qb for pairable cells
                const int ncp = misc[0];
                const int G = min(32, floor_pow2(NT / max(ncp, 1)));
                const int gsh = 31 - __clz(G);
                const int items = ncp << gsh;
                const int umax = min(MAXLOOP, d - 2 - (TURN + 1));
                const int ncand = umax >= 0 ? st->ncand_upto[umax] : 0;
                for (int base = tid - lane; base < items; base += NT) {
                    const int item = base + lane;
                    const bool active = item < items;
                    double acc = 0.;
                    int i = 0, j = 0, type = 0;
                    if (active) {
                        i = list[item >> gsh];
                        j = i + d;
                        type = ctype[i];
                        const int gl = item & (G - 1);
                        const int si1 = S[i + 1], sj1 = S[j - 1];
                        const int mi = mm_idx(type, si1, sj1);
                        const double oG = st->mmI[mi], o1 = st->mm1n[mi], oB = type > 2 ? st->expTermAU : 1.;
                        for (int ci = gl; ci < ncand; ci += G) {
                            const int cd = st->cand[ci];
                            const int u1 = cd & 31, u2 = (cd >> 5) & 31, cls = cd >> 10;
                            const int p = i + 1 + u1, q = j - 1 - u2;
                            if (cls != PCLS_TABLE) {
                                const double v = ring[cls * PRING * W + st->rowoff[u1 + u2] + p];
                                const double o = cls == PCLS_GENERIC ? oG : (cls == PCLS_1N ? o1 : oB);
                                acc += v * st->fac[ci] * o;
                                continue;
                            }
                            const double qpq = qb[TRI(q - p, p)];
                            if (qpq != 0.) {
                                const int t2 = rtype_of(pair_type(S[p], S[q]));
                                double z = x_intloop(c, u1, u2, type, t2, si1, sj1, S[p - 1], S[q + 1]) * scale[u1 + u2 + 2];
                                if (u1 == 0 && u2 == 0) z *= x_sc_stack(c, i, j, p, q);
                                acc += qpq * z;
                            }
                        }
                        // multiloop: sum_k qm[i+1,k-1] * qm1[k,j-1]
                        double ml = 0., ml2 = 0.;
                        {
                            const double *a = qmR + RM(i + 1, 0) - 1, *b = qm1C + CM(0, j - 1);   // a[k] = qm[i+1][k-1], b[k] = qm1[k][j-1]
                            int k = i + 2 + TURN + 1 + gl;
                            for (; k + G <= j - 2 - TURN; k += 2 * G) {
                                ml = fma(a[k], b[k], ml);
                                ml2 = fma(a[k + G], b[k + G], ml2);
                            }
                            if (k <= j - 2 - TURN) ml = fma(a[k], b[k], ml);
                        }
                        ml += ml2;
                        acc += ml * closing * x_mlstem(*st, rtype_of(type), sj1, si1) * scale[2];
                    }
                    acc = group_sum(acc, G);
                    if (active && (item & (G - 1)) == 0) {
                        const double qv = acc + x_hairpin(c, i, j, type) * scale[d + 1];
                        qb[tri_d + i] = qv;
                        double vG = 0., v1 = 0., vB = 0.;
                        if (i > 0 && j < W - 1) {  // (i,j) as the inner pair of an enclosing loop
                            const int t2 = rtype_of(type);
                            const int m2 = mm_idx(t2, S[j + 1], S[i - 1]);
                            vG = qv * st->mmI[m2];
                            v1 = qv * st->mm1n[m2];
                            vB = t2 > 2 ? qv * st->expTermAU : qv;
                        }
                        ring[ring_row + i] = vG;
                        ring[PRING * W + ring_row + i] = v1;
                        ring[2 * PRING * W + ring_row + i] = vB;
                    }
                }
            }
            __syncthreads();
            {   // qm1, qm for every cell
                const int G = min(32, floor_pow2(NT / ncells));
                const int gsh = 31 - __clz(G);
                const int items = ncells << gsh;
                for (int base = tid - lane; base < items; base += NT) {
                    const int item = base + lane;
                    const bool active = item < items;
                    double acc = 0.;
                    int i = 0, j = 0;
                    if (active) {
                        i = item >> gsh;
                        j = i + d;
                        // sum_{k=i+1}^{j-TURN-1} (qm[i,k-1] + eMLb[k-i]) * qm1[k,j]
                        const double *a = qmR + RM(i, 0) - 1, *b = qm1C + CM(0, j);   // a[k] = qm[i][k-1], b[k] = qm1[k][j]
                        double acc2 = 0.;
                        int k = i + 1 + (item & (G - 1));
                        for (; k + G <= j - TURN - 1; k += 2 * G) {
                            const double l0 = eMLb[k - i] + (k - 1 - i > TURN ? a[k] : 0.);
                            const double l1 = eMLb[k + G - i] + (k + G - 1 - i > TURN ? a[k + G] : 0.);
                            acc = fma(l0, b[k], acc);
                            acc2 = fma(l1, b[k + G], acc2);
                        }
                        if (k <= j - TURN - 1) acc = fma(eMLb[k - i] + (k - 1 - i > TURN ? a[k] : 0.), b[k], acc);
                        acc += acc2;
                    }
                    acc = group_sum(acc, G);
                    if (active && (item & (G - 1)) == 0) {
                        double v = (d - 1 > TURN) ? qm1C[CM(i, j - 1)] * eMLb[1] : 0.;
                        const int t = ctype[i];
                        if (t) v += qb[tri_d + i] * x_mlstem(*st, t, i > 0 ? S[i - 1] : -1, j < W - 1 ? S[j + 1] : -1);
                        qm1C[CM(i, j)] = v;
                        qmR[RM(i, j)] = acc + v;
                        qmC[CM(i, j)] = acc + v;
                    }
                }
            }
            __syncthreads();
        }

        // ================= exterior prefix / suffix sums (one warp) =================
        if (tid < 32) {
            if (lane == 0) {
                q5[0] = 1.;
                q3[W] = 1.;
            }
            __syncwarp();
            for (int len = 1; len <= W; len++) {
                const int j = len - 1;
                double acc = 0.;
                for (int i = lane; i <= j - TURN - 1; i += 32) {
                    const double q = qb[TRI(j - i, i)];
                    if (q != 0.)
                        acc += q5[i] * q *
                               x_extloop(*st, pair_type(S[i], S[j]), i > 0 ? S[i - 1] : -1, j < W - 1 ? S[j + 1] : -1);
                }
                acc = group_sum(acc, 32);
                if (lane == 0) q5[len] = q5[len - 1] * scale[1] + acc;
                __syncwarp();
            }
            for (int i = W - 1; i >= 0; i--) {
                double acc = 0.;
                for (int j = i + TURN + 1 + lane; j < W; j += 32) {
                    const double q = qb[TRI(j - i, i)];
                    if (q != 0.)
                        acc += q * q3[j + 1] *
                               x_extloop(*st, pair_type(S[i], S[j]), i > 0 ? S[i - 1] : -1, j < W - 1 ? S[j + 1] : -1);
                }
                acc = group_sum(acc, 32);
                if (lane == 0) q3[i] = q3[i + 1] * scale[1] + acc;
                __syncwarp();
            }
        }
        __syncthreads();
        const double Z = q5[W];

        // ================= outside =================
        double ed_local = 0.;
        for (int d = W - 1; d > TURN; d--) {
            const int ncells = W - d;
            const int tri_d = tri_off(d, W);
            const int G = min(32, floor_pow2(NT / ncells));
            const int gsh = 31 - __clz(G);
            const int items = ncells << gsh;
            if (tid < 32) st->rowoff[tid] = ((d + 2 + tid) % PRING) * W;
            __syncthreads();
            const int ring_row = (d % PRING) * W;
            // P[k,l]: exterior + enclosing interior loops + enclosing multiloops
            for (int base = tid - lane; base < items; base += NT) {
                const int item = base + lane;
                const bool active = item < items;
                double acc = 0.;
                int k = 0, l = 0, tkl = 0;
                double qkl = 0.;
                if (active) {
                    k = item >> gsh;
                    l = k + d;
                    qkl = qb[tri_d + k];
                    if (qkl != 0.) {
                        const int gl = item & (G - 1);
                        tkl = pair_type(S[k], S[l]);
                        const int t2 = rtype_of(tkl);
                        if (k > 0 && l < W - 1) {
                            const int sp1 = S[k - 1], sq1 = S[l + 1];
                            const int umax = min(MAXLOOP, W - 3 - d);
                            const int ncand = umax >= 0 ? st->ncand_upto[umax] : 0;
                            const int m2 = mm_idx(t2, sq1, sp1);
                            const double iG = st->mmI[m2], i1 = st->mm1n[m2], iB = t2 > 2 ? st->expTermAU : 1.;
                            for (int ci = gl; ci < ncand; ci += G) {
                                const int cd = st->cand[ci];
                                const int u1 = cd & 31, u2 = (cd >> 5) & 31, cls = cd >> 10;
                                const int i = k - 1 - u1, j = l + 1 + u2;
                                if (i < 0 || j > W - 1) continue;
                                if (cls != PCLS_TABLE) {
                                    const double v = ring[cls * PRING * W + st->rowoff[u1 + u2] + i];
                                    const double o = cls == PCLS_GENERIC ? iG : (cls == PCLS_1N ? i1 : iB);
                                    acc += v * st->fac[ci] * o;
                                    continue;
                                }
                                const double pij = Pm[TRI(j - i, i)];
                                if (pij > 0.) {
                                    const int tij = pair_type(S[i], S[j]);
                                    double z = x_intloop(c, u1, u2, tij, t2, S[i + 1], S[j - 1], sp1, sq1) * scale[u1 + u2 + 2];
                                    if (u1 == 0 && u2 == 0) z *= x_sc_stack(c, i, j, k, l);
                                    acc += pij * z;
                                }
                            }
                            // multiloop closed by (i,j), i < k, j > l
                            double ml = 0., mlb = 0.;
                            {
                                const double *x1c = X1C + CM(0, l), *x2c = X2C + CM(0, l), *qc = qmC + CM(1, k - 1);   // qc[i] = qm[i+1][k-1]
                                int i = gl;
                                for (; i + G <= k - 1; i += 2 * G) {
                                    const double a0 = x1c[i], a1 = x1c[i + G];
                                    ml = fma(a0, eMLb[k - 1 - i], ml);
                                    mlb = fma(a1, eMLb[k - 1 - i - G], mlb);
                                    if (k - 2 - i > TURN) ml = fma(a0 + x2c[i], qc[i], ml);
                                    if (k - 2 - i - G > TURN) mlb = fma(a1 + x2c[i + G], qc[i + G], mlb);
                                }
                                if (i <= k - 1) {
                                    const double a0 = x1c[i];
                                    ml = fma(a0, eMLb[k - 1 - i], ml);
                                    if (k - 2 - i > TURN) ml = fma(a0 + x2c[i], qc[i], ml);
                                }
                            }
                            ml += mlb;
                            acc += ml * x_mlstem(*st, tkl, sp1, sq1) * scale[2];
                        }
                        if (gl == 0)
                            acc += q5[k] * q3[l + 1] / Z *
                                   x_extloop(*st, tkl, k > 0 ? S[k - 1] : -1, l < W - 1 ? S[l + 1] : -1);
                    }
                }
                acc = group_sum(acc, G);
                if (active && (item & (G - 1)) == 0) {
                    Pm[tri_d + k] = acc;
                    {   // (k,l) as the OUTER pair of loops enclosing pairs on shorter diagonals
                        double vG = 0., v1 = 0., vB = 0.;
                        if (acc != 0.) {
                            const int mo = mm_idx(tkl, S[k + 1], S[l - 1]);
                            vG = acc * st->mmI[mo];
                            v1 = acc * st->mm1n[mo];
                            vB = tkl > 2 ? acc * st->expTermAU : acc;
                        }
                        ring[ring_row + k] = vG;
                        ring[PRING * W + ring_row + k] = v1;
                        ring[2 * PRING * W + ring_row + k] = vB;
                    }
                    double pm = 0.;
                    if (qkl != 0. && k + 1 < W && l >= 1)
                        pm = acc * closing * x_mlstem(*st, rtype_of(tkl), S[l - 1], S[k + 1]);
                    PMR[RM(k, l)] = pm;
                    const double p = acc * qkl;
                    ed_local += p * (1. - p);
                    if (p > 0.5) {
                        cen[k] = (int16_t)(l + 1);
                        cen[l] = (int16_t)(k + 1);
                    }
                    if (L.bpp) L.bpp[((long long)fold * W + k) * W + l] = p;
                }
            }
            __syncthreads();
            // X1[i,l] = sum_{j>=l+2} PM[i,j] qm[l+1,j-1];  X2[i,l] = X2[i,l+1] eMLb[1] + PM[i,l+1]
            for (int base = tid - lane; base < items; base += NT) {
                const int item = base + lane;
                const bool active = item < items;
                double acc = 0.;
                int i = 0, l = 0;
                if (active) {
                    i = item >> gsh;
                    l = i + d;
                    const double *a = PMR + RM(i, 0), *b = qmR + RM(l + 1, 0) - 1;   // a[j] = PM[i][j], b[j] = qm[l+1][j-1]
                    double acc2 = 0.;
                    int j = l + 2 + TURN + 1 + (item & (G - 1));
                    for (; j + G < W; j += 2 * G) {
                        acc = fma(a[j], b[j], acc);
                        acc2 = fma(a[j + G], b[j + G], acc2);
                    }
                    if (j < W) acc = fma(a[j], b[j], acc);
                    acc += acc2;
                }
                acc = group_sum(acc, G);
                if (active && (item & (G - 1)) == 0) {
                    X1C[CM(i, l)] = acc;
                    double x2 = 0.;
                    if (l + 1 < W) x2 = X2C[CM(i, l + 1)] * eMLb[1] + PMR[RM(i, l + 1)];
                    X2C[CM(i, l)] = x2;
                }
            }
            __syncthreads();
        }

        // ================= ED, centroid =================
        for (int o = 16; o; o >>= 1) ed_local += __shfl_xor_sync(0xffffffffu, ed_local, o);
        if (lane == 0) red[tid >> 5] = ed_local;
        __syncthreads();
        if (tid == 0) {
            double s = 0.;
            for (int w = 0; w < NT / 32; w++) s += red[w];
            const double dG = (-log(Z) - W * log(st->pf_scale)) * st->kT / 1000.;
            L.ed[fold] = 2. * s;
            L.dG[fold] = dG;
            if (L.n_out_of_range && !(isfinite(dG) && isfinite(2. * s))) atomicAdd(L.n_out_of_range, 1);
        }
        for (int k = tid; k < W; k += NT) L.centroid[(long long)fold * W + k] = cen[k];
        if constexpr (PAIRPROB) {
            double s = 0.;   // as thread 0 formed it
            for (int w = 0; w < NT / 32; w++) s += red[w];
            const double dG = (-log(Z) - W * log(st->pf_scale)) * st->kT / 1000.;
            if (isfinite(dG) && isfinite(2. * s)) {
                long long *rows = pp.table + (pp.row0 + (long long)fold * pp.step) * W;
                for (int i = tid; i < W; i += NT)
                    pp_commit_row(rows, i, W, [&](int k, int l) { return Pm[TRI(l - k, k)] * qb[TRI(l - k, k)]; });
            }
        }
        __syncthreads();
    }
#undef TRI
#undef RM
#undef CM
}

size_t pf_smem_bytes(int W) {
    size_t b = (sizeof(PfSmall) + 15) & ~(size_t)15;
    b += sizeof(double) * ((std::max(W, MAXLOOP) + 4) + (W + 4) + 2 * (W + 2) + 8);
    b += sizeof(int) * ((W + 2) + 4 + (W + 2));
    b += sizeof(int16_t) * 3 * W + 3 * (W + 4);
    return (b + 15) & ~(size_t)15;
}

}  // namespace

size_t pf_scratch_doubles_per_cta(int W, bool pairprob) {
    const size_t a = 2 * ((size_t)W * (W + 1) / 2) + 6 * (size_t)W * W + 3 * (size_t)PRING * W, b = pf2_scratch_doubles_per_cta(pairprob);
    return a > b ? a : b;
}

int pf_grid_size(int W, int n_sm, int n_fold) {
    // resident CTAs: the kernel waits on L2, occupancy is what hides it (registers allow SFB_PF_MINB, shared memory less
    // for long windows)
    long long per_sm = (long long)((227 * 1024) / (pf_smem_bytes(W) + 1024));
    if (per_sm > SFB_PF_MINB) per_sm = SFB_PF_MINB;
    if (per_sm < 1) per_sm = 1;
    long long g = (long long)n_sm * per_sm;
    if (g > n_fold) g = n_fold;
    return (int)g;
}

void launch_pf(const PfLaunch &L, const MfeTables *d_mfe, const PfTables *d_pf, int n_sm, cudaStream_t stream,
               int *n_launches, const PairProbCommit &pp) {
    if (L.n_fold <= 0) return;
    if (pf2_supports(L)) {   // unconstrained windows up to 120 nt: shared-memory kernel (pf2.cu)
        launch_pf2(L, d_mfe, d_pf, n_sm, stream, n_launches, pp);
        return;
    }
    size_t smem = pf_smem_bytes(L.W);
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(pf_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024));
        cudaFuncSetAttribute(pf_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024));
        configured = true;
    }
    int grid = pf_grid_size(L.W, n_sm, L.n_fold);
    if (pp.table)
        pf_kernel<true><<<grid, NT, smem, stream>>>(L, d_mfe, d_pf, pp);
    else
        pf_kernel<false><<<grid, NT, smem, stream>>>(L, d_mfe, d_pf, pp);
    if (n_launches) (*n_launches)++;
}

}  // namespace sfb
