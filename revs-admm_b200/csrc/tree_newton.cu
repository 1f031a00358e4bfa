// Operator QP of a LARGE radial zone: one CTA per (zone, hour) column, every linear-algebra step on the feeder tree.
//
// Reference: class Utility (lpsolver.py:163-238) hands  min 1/2 |g - z|^2, g >= 0, R g <= u  with the dense
// R = 2 F D F^T (compute_Rmat, lpsolver.py:17-26) of ALL residences of the graph to Gurobi; nothing there limits the
// number of rows that bind.  The dense kernels of this library (utility_qp*.cu) keep the model Hessian H_AA of the
// binding rows in shared memory and stop at 128 of them; an unsplit 10k-home feeder under tight limits binds several
// hundred per hour (BASELINE.json config 3).  Here neither R nor H is ever formed:
//
//   * PRODUCT  mu = R x:   Lam_k = x_k + sum_{children} Lam_c  (leaves -> root),  mu_k = mu_parent + rho_k Lam_k
//     (root -> leaves), rho_k = 2 r_k.  One pass up, one pass down, a barrier per tree level.
//   * SOLVE of one active-set guess (rows A at their limit on the piece F = {g > 0}):
//         R_AF (z_F - R_FA x_A) - s x_A = t_A          <=>   (R_AF R_FA + s I) x_A = R_AF z_F - t_A
//     is a two-point boundary problem on the same tree: the subtree below the edge above node k answers its parent's
//     (mu_p, v_p) with an affine map (Lam_k, f_k) = M_k (mu_p, v_p) + m_k, the maps of the children add, and a node is
//     eliminated by one 2 x 2 solve.  Pass up: M, m and the back-substitution map of every node; pass down: mu, v, x.
//     O(nodes) per guess for ANY number of binding rows, exact to rounding (symmetric quasi-definite elimination).
//
// The iteration around them is the one of oracle.project_voltage / utility_qp.cu: KKT test on the exact voltages, working
// rows W = {lam > 0} u {violated}, the quadratic piece minimised exactly over lam_W >= 0 by a primal-dual active set
// (every guess = one tree solve), line search of the true dual on the segment, Levenberg-Marquardt safeguard.  The QP is
// strictly convex in g, so the result is the same unique point the dense path and the reference's solver return.
//
// Two things make the elimination robust on real feeders (the reference's network 121144 has primary edges of 1e-20 and
// idle homes at the end of laterals):
//   * edges of negligible resistance are contracted on the host, so a node may carry several residences; their voltage
//     rows are identical, the node has ONE row and one multiplier, its homes differ only in z and in being on the piece;
//   * an active row whose subtree holds no home of the piece has no leverage of its own (nothing below it flows): its
//     2 x 2 pivot would be the shift alone.  Such a node PINS its parent instead -- "your voltage is my target" -- and
//     hands its dual flow up as the parent's unknown; pins travel up idle chains, the tightest of several pins on a
//     node is kept, the others (duplicate rows) sit the guess out as plain nodes.
//
// Layout: the nodes of a zone are renumbered breadth-first (a level = a contiguous range, the children of a node
// contiguous in the next level), static arrays per zone, ~300 bytes of per-node work arrays per column in global memory
// (L2-resident; plain loads -- the arrays are written by other threads of the CTA, never through the read-only path).
// A level pass is a chain of dependent steps, one per tree level (141 for the 10k-home feeder), so what matters is the
// latency of ONE step: the messages between adjacent levels (8 doubles per node up, 3 down) travel through a
// double-buffered shared-memory exchange, everything a node needs that does not depend on the neighbouring level is
// prefetched one level ahead into registers, results go to global memory as fire-and-forget stores, and all per-home
// work (gathers, clipping, sums) happens in flat loops outside the level passes.  A step is then a barrier, a few
// shared-memory reads and ~40 dependent FP64 operations.  numpy model of this file: tests/tree_newton_ref.py.
#include <math_constants.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "kernels.cuh"

namespace revs {

namespace {

constexpr int kNtThreads = 256;
constexpr int kXCap = 512;                         // nodes of a level whose messages travel through shared memory (the rest: global)
constexpr int kLvlCap = 1024;                      // level offsets cached in shared memory
constexpr double kArcMinN = 9.5367431640625e-07;   // 2^-20
constexpr int kPdasMaxN = 24;
constexpr double kHessShiftN = 1e-20;              // structural singularities are handled by the pins, not by the shift
constexpr double kLmShiftN = 1e-12;                // base shift of the Levenberg-Marquardt safeguard
constexpr double kPhiNoiseN = 1e-14;
constexpr double kDegTolN = 1e-9;                  // |d(flow of the subtree)/d(mu)| below this: no home of the piece below the row
constexpr double kPdasSlackN = 1e-13;              // a row off the guess re-enters when violated by more than this fraction of u
constexpr double kContractRelN = 1e-10;            // edges below this fraction of the largest root-to-node resistance are contracted
constexpr int kOuterMaxN = 200;

enum : int { kRes = 1, kW = 2, kA = 4, kPin = 8, kEff = 16 };

struct Col {                 // work arrays of one column
    double *z, *g, *gn;                                                     // per home (node-sorted order)
    double *lam, *ln, *x, *mu, *v, *acc, *gr, *mrest, *nf, *zf, *gs, *xig, *tauP, *cP, *tau;   // per node
    double4 *M, *K, *P4;     // message of the subtree / back-substitution as the node acts / pin record
    double2 *m, *kv;
    int *fl, *src, *kept;
};

struct Zone {
    int nn, nlev, n;
    const int* lvl;          // [nlev + 1] (shared-memory copy when it fits)
    const int* parent;
    const int2* child;       // {first child, number of children}
    const int2* homes;       // {first home, number of homes} in the node-sorted home order
    const double* rho;
    const int* hlist;        // [n] home index inside the zone of every node-sorted position
    const int* hnode;        // [n] node of every node-sorted position
};

struct Xch { double (*up)[8]; };     // shared-memory exchange: [2][kXCap][8]

__device__ __forceinline__ double block_sum(double v, double* red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < kNtThreads / 32; ++i) t += red[i];
    return t;
}
__device__ __forceinline__ double block_max(double v, double* red) {
    v = warp_max(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    double t = red[0];
#pragma unroll
    for (int i = 1; i < kNtThreads / 32; ++i) t = fmax(t, red[i]);
    return t;
}
__device__ __forceinline__ int block_count(bool p, int* red) {
    const unsigned b = __ballot_sync(0xffffffffu, p);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[w] = __popc(b);
    __syncthreads();
    int t = 0;
#pragma unroll
    for (int i = 0; i < kNtThreads / 32; ++i) t += red[i];
    return t;
}

// ---- product: out = R x, x given per node in `src` (a global array).  Leaves -> root: acc = subtree sums (tree_sums);
// root -> leaves: out_k = out_parent + rho_k acc_k.  Messages through X (one double per node), inputs prefetched a level ahead.
template <bool MAX>
__device__ __forceinline__ void tree_sums(const Zone& Z, const Xch& X, const double* src, double* acc) {
    const int tid = threadIdx.x;
    {
        int l = Z.nlev - 1;
        int kn = Z.lvl[l] + tid;
        bool hn = kn < Z.lvl[l + 1];
        int2 chn = hn ? Z.child[kn] : make_int2(0, 0);
        double sn = hn ? src[kn] : 0.0;
        for (; l >= 0; --l) {
            const int lo = Z.lvl[l], hi = Z.lvl[l + 1];
            const int2 ch0 = chn;
            const double s0 = sn;
            if (l > 0) {
                kn = Z.lvl[l - 1] + tid;
                hn = kn < lo;
                chn = hn ? Z.child[kn] : make_int2(0, 0);
                sn = hn ? src[kn] : 0.0;
            }
            double(*bc)[8] = X.up + ((l + 1) & 1) * kXCap;
            double(*bo)[8] = X.up + (l & 1) * kXCap;
            for (int k = lo + tid; k < hi; k += kNtThreads) {
                const bool first = k == lo + tid;
                const int2 ch = first ? ch0 : Z.child[k];
                double a = first ? s0 : src[k];
                for (int j = 0; j < ch.y; ++j) {
                    const int cl = ch.x + j - hi;
                    const double ac = cl < kXCap ? bc[cl][0] : acc[ch.x + j];
                    a = MAX ? fmax(a, ac) : a + ac;
                }
                acc[k] = a;
                if (k - lo < kXCap) bo[k - lo][0] = a;
            }
            __syncthreads();
        }
    }
}
__device__ __forceinline__ void tree_product(const Zone& Z, const Xch& X, const double* src, double* acc, double* out) {
    const int tid = threadIdx.x;
    tree_sums<false>(Z, X, src, acc);
    {
        int kn = Z.lvl[0] + tid;
        bool hn = kn < Z.lvl[1];
        int pn = hn ? Z.parent[kn] : -1;
        double rn = hn ? Z.rho[kn] : 0.0, an = hn ? acc[kn] : 0.0;
        for (int l = 0; l < Z.nlev; ++l) {
            const int lo = Z.lvl[l], hi = Z.lvl[l + 1];
            const int p0 = pn;
            const double r0 = rn, a0 = an;
            if (l + 1 < Z.nlev) {
                kn = hi + tid;
                hn = kn < Z.lvl[l + 2];
                pn = hn ? Z.parent[kn] : -1;
                rn = hn ? Z.rho[kn] : 0.0;
                an = hn ? acc[kn] : 0.0;
            }
            const int lop = l > 0 ? Z.lvl[l - 1] : 0;
            double(*bp)[8] = X.up + ((l + 1) & 1) * kXCap;       // == buffer (l - 1) & 1
            double(*bo)[8] = X.up + (l & 1) * kXCap;
            for (int k = lo + tid; k < hi; k += kNtThreads) {
                const bool first = k == lo + tid;
                const int p = first ? p0 : Z.parent[k];
                const double r = first ? r0 : Z.rho[k], a = first ? a0 : acc[k];
                double op = 0.0;
                if (p >= 0) op = p - lop < kXCap ? bp[p - lop][0] : out[p];
                const double o = fma(r, a, op);
                out[k] = o;
                if (k - lo < kXCap) bo[k - lo][0] = o;
            }
            __syncthreads();
        }
    }
}

// phi(lam_src) = 1/2 |[z - R lam]_+|^2 + u sum(lam); the iterate [z - R lam]_+ goes to gout (per home)
__device__ __forceinline__ double eval_phi(const Zone& Z, const Xch& X, const Col& C, double u, const double* lsrc, double* gout, double* red) {
    tree_product(Z, X, lsrc, C.acc, C.mu);
    double part = 0.0;
    for (int j = threadIdx.x; j < Z.n; j += kNtThreads) {
        const double gk = fmax(C.z[j] - C.mu[Z.hnode[j]], 0.0);
        gout[j] = gk;
        part = fma(0.5 * gk, gk, part);
    }
    for (int k = threadIdx.x; k < Z.nn; k += kNtThreads) part = fma(u, lsrc[k], part);
    return block_sum(part, red);
}

// per node: sum of g over its homes (gs), number of homes on the piece and sum of their targets (nf, zf)
__device__ __forceinline__ void node_sums(const Zone& Z, const Col& C, bool use_rest) {
    for (int k = threadIdx.x; k < Z.nn; k += kNtThreads) {
        const int2 hh = Z.homes[k];
        double gsum = 0.0, nf = 0.0, zf = 0.0;
        if (hh.y) {
            const double rest = use_rest ? C.mrest[k] : 0.0;
            for (int j = hh.x; j < hh.x + hh.y; ++j) {
                const double gj = C.g[j];
                gsum += gj;
                if (gj > 0.0) { nf += 1.0; zf += C.z[j] - rest; }
            }
        }
        C.gs[k] = gsum; C.nf[k] = nf; C.zf[k] = zf;
    }
    __syncthreads();
}

struct Elim { double4 M, K; double2 m, kv; };

// node that enforces no row:  (mu, v) = K p + kv,  (Lam, f) = M p + m
__device__ __forceinline__ Elim elim_plain(double S00, double S01, double S10, double S11, double s0, double s1, double r) {
    const double a = 1.0 - r * S00, b = -r * S01, c = -r * S10, d = 1.0 - r * S11;
    const double inv = 1.0 / (a * d - b * c);
    const double i00 = d * inv, i01 = -b * inv, i10 = -c * inv, i11 = a * inv;
    const double q0 = r * s0, q1 = r * s1;
    const double k0 = i00 * q0 + i01 * q1, k1 = i10 * q0 + i11 * q1;
    Elim e;
    e.K = make_double4(i00, i01, i10, i11);
    e.kv = make_double2(k0, k1);
    e.M = make_double4(S00 * i00 + S01 * i10, S00 * i01 + S01 * i11, S10 * i00 + S11 * i10, S10 * i01 + S11 * i11);
    e.m = make_double2(S00 * k0 + S01 * k1 + s0, S10 * k0 + S11 * k1 + s1);
    return e;
}
// node with an effective row  v - s xi = t:  (mu, xi) = K p + kv
__device__ __forceinline__ Elim elim_active(double S00, double S01, double S10, double S11, double s0, double s1, double r, double t, double s) {
    const double a = 1.0 - r * S00, c = -r * S10;
    const double b = -r * fma(S01, s, 1.0), d = s * (1.0 - r * S11);
    const double q0 = r * fma(S01, t, s0), q1 = fma(r, fma(S11, t, s1), -t);
    const double C01 = fma(S01, s, 1.0), C11 = S11 * s, c00 = fma(S01, t, s0), c01 = fma(S11, t, s1);
    const double inv = 1.0 / (a * d - b * c);
    const double i00 = d * inv, i01 = -b * inv, i10 = -c * inv, i11 = a * inv;
    const double k0 = i00 * q0 + i01 * q1, k1 = i10 * q0 + i11 * q1;
    Elim e;
    e.K = make_double4(i00, i01, i10, i11);
    e.kv = make_double2(k0, k1);
    e.M = make_double4(S00 * i00 + C01 * i10, S00 * i01 + C01 * i11, S10 * i00 + C11 * i10, S10 * i01 + C11 * i11);
    e.m = make_double2(S00 * k0 + C01 * k1 + c00, S10 * k0 + C11 * k1 + c01);
    return e;
}

// One active-set guess: x on the node rows flagged kA with v - s x = u - s lam on the rows that take part, for
// g_h = z_h - mu[node(h)] on the homes of the piece (C.nf / C.zf, see node_sums), 0 elsewhere, v = R g.
// Results: C.x (0 off A), C.v (voltages of the guess).
// Message of node k to its parent (8 doubles): M (4), m (2), voltage it pins the parent to (inf: none), its constant flow.
struct UpIn { int2 ch; int fl; double r, lam, nf, zf; int parent; };

__device__ __forceinline__ UpIn load_up(const Zone& Z, const Col& C, int k) {
    UpIn i;
    i.ch = Z.child[k]; i.fl = C.fl[k]; i.r = Z.rho[k]; i.lam = C.lam[k]; i.nf = C.nf[k]; i.zf = C.zf[k]; i.parent = Z.parent[k];
    return i;
}
struct DnIn { int parent, fl, kept, src; double4 K; double2 kv; double tau, lam; };

__device__ __forceinline__ DnIn load_dn(const Zone& Z, const Col& C, int k) {
    DnIn i;
    i.parent = Z.parent[k]; i.fl = C.fl[k]; i.kept = C.kept[k]; i.src = C.src[k];
    i.K = C.K[k]; i.kv = C.kv[k]; i.tau = C.tau[k]; i.lam = C.lam[k];
    return i;
}

__device__ __forceinline__ void tree_solve(const Zone& Z, const Xch& X, const Col& C, double u, double s) {
    const int tid = threadIdx.x;
    {
        int l = Z.nlev - 1;
        int kn = Z.lvl[l] + tid;
        UpIn nx{};
        if (kn < Z.lvl[l + 1]) nx = load_up(Z, C, kn);
        for (; l >= 0; --l) {
            const int lo = Z.lvl[l], hi = Z.lvl[l + 1];
            const UpIn c0 = nx;
            if (l > 0) {
                kn = Z.lvl[l - 1] + tid;
                if (kn < lo) nx = load_up(Z, C, kn);
            }
            double(*bc)[8] = X.up + ((l + 1) & 1) * kXCap;
            double(*bo)[8] = X.up + (l & 1) * kXCap;
            for (int k = lo + tid; k < hi; k += kNtThreads) {
                const UpIn in = k == lo + tid ? c0 : load_up(Z, C, k);
                int fl = in.fl & ~(kPin | kEff);
                double tk = CUDART_INF;
                int sk = -2;
                if (fl & kA) { tk = u - s * in.lam; sk = -1; }
                // the tightest pin among the children (and the own row) is the effective row of this node
                for (int j = 0; j < in.ch.y; ++j) {
                    const int c = in.ch.x + j, cl = c - hi;
                    const double tp = cl < kXCap ? bc[cl][6] : C.tauP[c];
                    if (tp < tk) { tk = tp; sk = c; }
                }
                double n00 = 0.0, n01 = 0.0, n10 = 0.0, n11 = 0.0, n0 = 0.0, n1 = 0.0;   // every child as it acts without a kept pin
                double e00 = 0.0, e01 = 0.0, e10 = 0.0, e11 = 0.0, e0 = 0.0, e1 = 0.0;   // the kept pin replaced by its message: its constant flow
                for (int j = 0; j < in.ch.y; ++j) {
                    const int c = in.ch.x + j, cl = c - hi;
                    double q[8];
                    if (cl < kXCap) {
#pragma unroll
                        for (int e = 0; e < 8; ++e) q[e] = bc[cl][e];
                    } else {
                        const double4 Mc = C.M[c];
                        const double2 mc = C.m[c];
                        q[0] = Mc.x; q[1] = Mc.y; q[2] = Mc.z; q[3] = Mc.w; q[4] = mc.x; q[5] = mc.y; q[6] = C.tauP[c]; q[7] = C.cP[c];
                    }
                    n00 += q[0]; n01 += q[1]; n10 += q[2]; n11 += q[3]; n0 += q[4]; n1 += q[5];
                    if (c == sk) e1 += q[7];
                    else { e00 += q[0]; e01 += q[1]; e10 += q[2]; e11 += q[3]; e0 += q[4]; e1 += q[5]; }
                }
                n10 -= in.nf; e10 -= in.nf; n1 += in.zf; e1 += in.zf;
                Elim P = elim_plain(n00, n01, n10, n11, n0, n1, in.r);
                double4 Kact = P.K;
                double2 kvact = P.kv;
                double tauP = CUDART_INF, cP = 0.0;
                if (sk != -2) {
                    if (fabs(e10) < kDegTolN) {
                        // nothing below responds to the multiplier: the row pins the parent (no parent: it cannot bind)
                        if (in.parent < 0) sk = -2;
                        else {
                            cP = fma(e11, tk, e1);
                            tauP = tk - in.r * cP;
                            fl |= kPin;
                            C.P4[k] = make_double4(e00, e01, e0, cP);
                        }
                    } else {
                        P = elim_active(e00, e01, e10, e11, e0, e1, in.r, tk, s);
                        Kact = P.K; kvact = P.kv;
                        fl |= kEff;
                    }
                }
                if (k - lo < kXCap) {
                    double* o = bo[k - lo];
                    o[0] = P.M.x; o[1] = P.M.y; o[2] = P.M.z; o[3] = P.M.w; o[4] = P.m.x; o[5] = P.m.y; o[6] = tauP; o[7] = cP;
                } else {
                    C.M[k] = P.M; C.m[k] = P.m; C.tauP[k] = tauP; C.cP[k] = cP;
                }
                C.K[k] = Kact; C.kv[k] = kvact;
                C.tau[k] = tk;
                C.src[k] = sk;
                C.fl[k] = fl;
                C.kept[k] = 0;
                if (sk >= 0) C.kept[sk] = 1;          // (the child reset its flag one level earlier)
            }
            __syncthreads();
        }
    }
    {
        int kn = Z.lvl[0] + tid;
        DnIn nx{};
        if (kn < Z.lvl[1]) nx = load_dn(Z, C, kn);
        for (int l = 0; l < Z.nlev; ++l) {
            const int lo = Z.lvl[l], hi = Z.lvl[l + 1];
            const DnIn c0 = nx;
            if (l + 1 < Z.nlev) {
                kn = hi + tid;
                if (kn < Z.lvl[l + 2]) nx = load_dn(Z, C, kn);
            }
            const int lop = l > 0 ? Z.lvl[l - 1] : 0;
            double(*bp)[8] = X.up + ((l + 1) & 1) * kXCap;
            double(*bo)[8] = X.up + (l & 1) * kXCap;
            for (int k = lo + tid; k < hi; k += kNtThreads) {
                const DnIn in = k == lo + tid ? c0 : load_dn(Z, C, k);
                double mp = 0.0, vp = 0.0, Xi = 0.0;
                if (in.parent >= 0) {
                    const int pl = in.parent - lop;
                    if (pl < kXCap) { mp = bp[pl][0]; vp = bp[pl][1]; Xi = bp[pl][2]; }
                    else { mp = C.mu[in.parent]; vp = C.v[in.parent]; Xi = C.xig[in.parent]; }
                }
                double muk, vk, xi = 0.0;
                bool eff = false;
                if ((in.fl & kPin) && in.kept && !isnan(Xi)) {
                    const double4 P4 = C.P4[k];
                    muk = fma(Z.rho[k], Xi, mp);
                    vk = in.tau;
                    xi = Xi - fma(P4.x, muk, fma(P4.y, vk, P4.z));
                    eff = true;
                } else if (in.fl & kEff) {
                    muk = fma(in.K.x, mp, fma(in.K.y, vp, in.kv.x));
                    xi = fma(in.K.z, mp, fma(in.K.w, vp, in.kv.y));
                    vk = fma(s, xi, in.tau);
                    eff = true;
                } else {
                    muk = fma(in.K.x, mp, fma(in.K.y, vp, in.kv.x));
                    vk = fma(in.K.z, mp, fma(in.K.w, vp, in.kv.y));
                }
                const double xk = (eff && in.src == -1) ? xi : 0.0;
                const double xo = (eff && in.src >= 0) ? xi : CUDART_NAN;   // dual flow handed to the kept pin below (nan: no pin is enforced)
                if (k - lo < kXCap) { double* o = bo[k - lo]; o[0] = muk; o[1] = vk; o[2] = xo; }
                C.mu[k] = muk; C.v[k] = vk; C.xig[k] = xo; C.x[k] = xk;
            }
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(kNtThreads) tree_newton_kernel(NewtonParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double red[kNtThreads / 32];
    __shared__ int redi[kNtThreads / 32];
    __shared__ int slvl[kLvlCap + 1];
    Xch X;
    X.up = reinterpret_cast<double(*)[8]>(smem_raw);
    const int c = blockIdx.x;                       // column of the list: zone-major, hour-minor
    int zi = 0;
    while (zi + 1 < P.n_zones && c >= P.zones[zi + 1].col0) ++zi;
    const NewtonZone nz = P.zones[zi];
    const int t = c - nz.col0;
    Zone Z;
    Z.nn = nz.nn; Z.nlev = nz.nlev; Z.n = nz.n;
    Z.lvl = P.lvl + nz.lvl_off;
    if (nz.nlev <= kLvlCap) {
        for (int i = threadIdx.x; i <= nz.nlev; i += kNtThreads) slvl[i] = Z.lvl[i];
        Z.lvl = slvl;
    }
    Z.parent = P.parent + nz.node_off;
    Z.child = P.child + nz.node_off;
    Z.homes = P.homes + nz.node_off;
    Z.rho = P.rho + nz.node_off;
    Z.hlist = P.hlist + nz.home_off;
    Z.hnode = P.hnode + nz.home_off;
    const size_t wo = (size_t)nz.ws_off + (size_t)t * nz.wn, st = (size_t)P.ws_stride;
    Col C;
    {
        double* w = P.ws + wo;
        C.z = w; C.g = w + st; C.gn = w + 2 * st; C.lam = w + 3 * st; C.ln = w + 4 * st; C.x = w + 5 * st; C.mu = w + 6 * st;
        C.v = w + 7 * st; C.acc = w + 8 * st; C.gr = w + 9 * st; C.mrest = w + 10 * st; C.nf = w + 11 * st; C.zf = w + 12 * st;
        C.gs = w + 13 * st; C.xig = w + 14 * st; C.tauP = w + 15 * st; C.cP = w + 16 * st; C.tau = w + 17 * st;
    }
    C.M = P.ws4 + wo; C.K = C.M + st; C.P4 = C.K + st;
    C.m = P.ws2 + wo; C.kv = C.m + st;
    C.fl = P.wsi + wo; C.src = C.fl + st; C.kept = C.src + st;
    const int nn = Z.nn, n = Z.n;
    const double u = P.u, tol = P.tol;
    const FeederDev fd = P.feeders[nz.feeder];
    const size_t col = (size_t)t * P.Hp + fd.off;
    const double* z_col = P.z_t + col;
    double* lam_col = P.lam_t + col;
    double* g_col = P.g_t + col;
    const int colid = nz.feeder * P.T + t;

    for (int j = threadIdx.x; j < n; j += kNtThreads) C.z[j] = z_col[Z.hlist[j]];
    for (int k = threadIdx.x; k < nn; k += kNtThreads) {
        const int2 hh = Z.homes[k];
        double lk = 0.0;
        for (int j = hh.x; j < hh.x + hh.y; ++j) lk += fmax(lam_col[Z.hlist[j]], 0.0);
        C.lam[k] = lk;
        C.fl[k] = hh.y ? kRes : 0;
    }
    __syncthreads();
    const double scale = nz.scale;
    double f = eval_phi(Z, X, C, u, C.lam, C.g, red);
    double tau = 1.0;
    int its = 0, n_solves = 0, status = 0, n_act = 0;
    for (; its < kOuterMaxN; ++its) {
        // ---- exact voltages of the iterate: KKT residual, gradient of the dual, working rows W (= first guess A)
        node_sums(Z, C, false);
        tree_product(Z, X, C.gs, C.acc, C.v);
        double kk = 0.0;
        int nact = 0;
        for (int k = threadIdx.x; k < nn; k += kNtThreads) {
            const int fl = C.fl[k] & kRes;
            double grad = 0.0, viol = 0.0;
            if (fl) {
                const double lk = C.lam[k];
                grad = u - C.v[k];
                kk = fmax(kk, lk > 0.0 ? fabs(grad) : fmax(-grad, 0.0));
                viol = fmax(-grad, 0.0);
                nact += lk > 0.0;
            }
            C.fl[k] = fl;
            C.gr[k] = grad;
            C.ln[k] = viol;
        }
        const double kkt = block_max(kk, red);
        n_act = (int)block_sum((double)nact, red);
        double* tr = (P.dbg_trace && its < 16) ? P.dbg_trace + ((size_t)c * 16 + its) * 4 : nullptr;
        if (tr && threadIdx.x == 0) { tr[0] = kkt; tr[1] = 0; tr[2] = 0; tr[3] = n_act; }
        if (kkt < tol) { status = 1; break; }
        const double shift = kHessShiftN * scale + 1e-300;

        // ---- working rows (= first guess): the multipliers' support and the SKYLINE of the violated rows -- a violated row
        // enters when no row in the subtree of its parent is more violated.  Under a heavy shared drop thousands of rows are
        // violated by similar amounts and a hundred end up binding; holding the skyline repairs most of the others, what is
        // left is admitted by the next iteration (the KKT test above always runs over all rows).
        tree_sums<true>(Z, X, C.ln, C.acc);
        for (int k = threadIdx.x; k < nn; k += kNtThreads) {
            int fl = C.fl[k];
            if (fl & kRes) {
                const double viol = C.ln[k];
                const int p = Z.parent[k];
                if (C.lam[k] > 0.0 || (viol > 0.0 && viol >= C.acc[p >= 0 ? p : k])) fl |= kW | kA;
                C.fl[k] = fl;
            }
        }
        __syncthreads();

        // ---- exact minimiser of the piece over lam_W >= 0: primal-dual active set, one tree solve per guess
        bool ok = false;
        for (int guess = 0; guess < kPdasMaxN; ++guess) {
            tree_solve(Z, X, C, u, shift);
            ++n_solves;
            if (P.dbg_dump && c == P.dbg_dump_col && its == P.dbg_dump_outer && guess == P.dbg_dump_guess) {
                for (int k = threadIdx.x; k < nn; k += kNtThreads) {
                    P.dbg_dump[k] = C.x[k]; P.dbg_dump[nn + k] = C.v[k]; P.dbg_dump[2 * nn + k] = (double)C.fl[k];
                    P.dbg_dump[3 * nn + k] = C.lam[k]; P.dbg_dump[4 * nn + k] = C.nf[k]; P.dbg_dump[5 * nn + k] = C.zf[k];
                    P.dbg_dump[6 * nn + k] = C.mu[k]; P.dbg_dump[7 * nn + k] = (double)C.src[k];
                }
                __syncthreads();
            }
            bool bad = false;
            for (int k = threadIdx.x; k < nn; k += kNtThreads) {
                int fl = C.fl[k];
                if (!(fl & kW)) continue;
                if (fl & kA) { if (C.x[k] <= 0.0) { fl &= ~kA; bad = true; } }
                else if (u - C.v[k] - shift * C.lam[k] < -kPdasSlackN * u) { fl |= kA; bad = true; }
                C.fl[k] = fl;
            }
            if (block_count(bad, redi) == 0) { ok = true; break; }
        }
        if (tr && threadIdx.x == 0) tr[1] = ok ? n_solves : -n_solves;
        double fn = f;
        {
            // ---- line search of the dual on the segment lam -> minimiser (direction kept in x).  When the guesses did not
            // settle, the last one clipped to lam >= 0 still gives a feasible direction: it is tried before the safeguard.
            double sl = 0.0;
            for (int k = threadIdx.x; k < nn; k += kNtThreads) {
                double d = 0.0;
                if (C.fl[k] & kW) { d = fmax(C.x[k], 0.0) - C.lam[k]; sl = fma(C.gr[k], d, sl); }
                C.x[k] = d;
            }
            const double slope = block_sum(sl, red);
            const bool settled = ok;
            ok = false;
            for (double a = 1.0; slope < 0.0 && a >= (settled ? kArcMinN : 1.0 / 64.0); a *= 0.5) {
                for (int k = threadIdx.x; k < nn; k += kNtThreads) C.ln[k] = fmax(fma(a, C.x[k], C.lam[k]), 0.0);
                __syncthreads();
                fn = eval_phi(Z, X, C, u, C.ln, C.gn, red);
                if (fn <= f + 1e-4 * a * slope + kPhiNoiseN * fabs(f)) { ok = true; if (tr && threadIdx.x == 0) tr[2] = a; break; }
            }
        }
        if (!ok) {
            // ---- safeguard: projected-Newton arc step with a Levenberg-Marquardt shift; rows at (numerically) zero
            // multiplier with a positive gradient are held, the targets lose their contribution
            const double eps = fmin(1e-8, kkt);
            bool rest = false;
            for (int k = threadIdx.x; k < nn; k += kNtThreads) {
                int fl = C.fl[k] & ~kA;
                double held = 0.0;
                if (fl & kW) {
                    if (!(C.lam[k] <= eps && C.gr[k] > 0.0)) fl |= kA;
                    else if (C.lam[k] > 0.0) { rest = true; held = C.lam[k]; }
                }
                C.fl[k] = fl;
                C.ln[k] = held;
            }
            if (block_count(rest, redi) > 0) {
                tree_product(Z, X, C.ln, C.acc, C.mrest);
                node_sums(Z, C, true);
            }
            bool found = false;
            double a = 1.0;
            for (;;) {
                const double sg = kLmShiftN * tau * scale + 1e-300;
                tree_solve(Z, X, C, u, sg);
                ++n_solves;
                for (int k = threadIdx.x; k < nn; k += kNtThreads) {
                    const int fl = C.fl[k];
                    C.x[k] = (fl & kA) ? C.x[k] - C.lam[k] : ((fl & kW) ? -C.lam[k] : 0.0);
                }
                __syncthreads();
                for (a = 1.0; a >= kArcMinN; a *= 0.5) {
                    double sl = 0.0;
                    for (int k = threadIdx.x; k < nn; k += kNtThreads) {
                        const double lnk = fmax(fma(a, C.x[k], C.lam[k]), 0.0);
                        C.ln[k] = lnk;
                        if (C.fl[k] & kW) sl = fma(C.gr[k], lnk - C.lam[k], sl);
                    }
                    const double slope = block_sum(sl, red);
                    fn = eval_phi(Z, X, C, u, C.ln, C.gn, red);
                    if (fn <= f + 1e-4 * slope + kPhiNoiseN * fabs(f)) { found = true; break; }
                }
                if (found || tau > 1e40) break;
                tau *= 1e3;
            }
            if (tr && threadIdx.x == 0) tr[2] = -tau;
            if (!found) { status = 2; break; }
            if (a == 1.0) tau = fmax(1.0, tau / 10.0);
        }
        for (int k = threadIdx.x; k < nn; k += kNtThreads) C.lam[k] = C.ln[k];
        for (int j = threadIdx.x; j < n; j += kNtThreads) C.g[j] = C.gn[j];
        __syncthreads();
        f = fn;
    }
    // ---- persist (a column that did not reach the tolerance raises the error flag and leaves the stored iterate alone);
    // the multiplier of a node goes to its first home
    if (status == 1) {
        for (int j = threadIdx.x; j < n; j += kNtThreads) g_col[Z.hlist[j]] = C.g[j];
        for (int k = threadIdx.x; k < nn; k += kNtThreads) {
            const int2 hh = Z.homes[k];
            for (int j = 0; j < hh.y; ++j) lam_col[Z.hlist[hh.x + j]] = j == 0 ? C.lam[k] : 0.0;
        }
    }
    if (threadIdx.x == 0) {
        P.status[colid] = 1;
        P.inner_ok[colid] = 1;
        P.wcount[colid] = 0;
        if (P.dbg_col) { P.dbg_col[2 * c] = n_solves; P.dbg_col[2 * c + 1] = its; }
        if (status != 1) atomicAdd(P.noconv, 1);
        atomicAdd(P.newton_its, (unsigned long long)n_solves);
        atomicAdd(P.cols, 1ull);
        atomicMax(P.max_ws, n_act);
        atomicAdd(P.flops, (unsigned long long)((double)nn * (90.0 * n_solves + 8.0 * (its + 1))));
    }
}

constexpr int kNtSmem = 2 * kXCap * 8 * (int)sizeof(double);

}  // namespace

// ---- host: contraction of negligible edges, breadth-first numbering, homes of every node
void newton_build_zone(int n_nodes, const int* parent, const double* r, int n_res, const int* res_node, NewtonZoneHost& Z) {
    std::vector<double> cum(n_nodes, 0.0);
    double cmax = 0.0;
    for (int k = 0; k < n_nodes; ++k) { cum[k] = (parent[k] >= 0 ? cum[parent[k]] : 0.0) + r[k]; cmax = std::max(cmax, cum[k]); }
    std::vector<int> rep(n_nodes), nw0(n_nodes, -1), par;
    std::vector<double> rr;
    for (int k = 0; k < n_nodes; ++k) {
        const bool tiny = parent[k] >= 0 && r[k] <= kContractRelN * cmax;
        rep[k] = tiny ? rep[parent[k]] : k;
        if (!tiny) { nw0[k] = (int)par.size(); par.push_back(parent[k] >= 0 ? nw0[rep[parent[k]]] : -1); rr.push_back(r[k]); }
    }
    const int n = (int)par.size();
    std::vector<int> cres(n_res);
    for (int h = 0; h < n_res; ++h) cres[h] = nw0[rep[res_node[h]]];
    BfsTree B;
    bfs_tree(n, par.data(), n_res, cres.data(), B);
    Z.lvl = std::move(B.lvl);
    Z.parent = std::move(B.parent);
    Z.child0 = std::move(B.child0);
    Z.nchild = std::move(B.nchild);
    Z.home0 = std::move(B.res0);
    Z.nhome = std::move(B.nres);
    Z.hlist = std::move(B.res);
    Z.rho.resize(n);
    for (int i = 0; i < n; ++i) Z.rho[i] = 2.0 * rr[B.order[i]];
    Z.hnode.resize(n_res);
    for (int i = 0; i < n; ++i)
        for (int j = Z.home0[i]; j < Z.home0[i] + Z.nhome[i]; ++j) Z.hnode[j] = i;
    // scale of the shifts: mean over the residences of (row sum of R)^2 / n (a lower bound of the squared row norm)
    std::vector<double> acc(n, 0.0), mu(n, 0.0);
    for (int i = 0; i < n; ++i) acc[i] = (double)Z.nhome[i];
    for (int i = n - 1; i >= 0; --i) if (Z.parent[i] >= 0) acc[Z.parent[i]] += acc[i];
    double sc = 0.0;
    for (int i = 0; i < n; ++i) {
        mu[i] = (Z.parent[i] >= 0 ? mu[Z.parent[i]] : 0.0) + Z.rho[i] * acc[i];
        sc += Z.nhome[i] * mu[i] * mu[i];
    }
    Z.scale = n_res > 0 ? sc / ((double)n_res * (double)n_res) : 1.0;
    if (!(Z.scale > 0.0)) Z.scale = 1.0;
}

cudaError_t launch_tree_newton(const NewtonParams& P, int n_cols, cudaStream_t stream) {
    if (n_cols <= 0) return cudaSuccess;
    static std::atomic<unsigned long long> attr_done{0};
    if (first_use_on_device(attr_done)) {
        cudaError_t e = cudaFuncSetAttribute(tree_newton_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kNtSmem);
        if (e != cudaSuccess) return e;
    }
    tree_newton_kernel<<<n_cols, kNtThreads, kNtSmem, stream>>>(P);
    return cudaGetLastError();
}

}  // namespace revs
