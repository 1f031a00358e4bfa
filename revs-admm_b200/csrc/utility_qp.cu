// Operator (utility) sub-problem of the ADMM loop: one CTA per (feeder, hour) column.
//
// Reference: class Utility (lpsolver.py:163-238), a Gurobi QP over all residences and
// hours at once.  It separates over hours; each hour is the Euclidean projection of
//     z = (P_est + P_sch)/2 - Gamma/kappa
// onto { g >= 0,  R g <= u },  u = vhigh^2 - vset^2  (Gurobi's default lb=0; the vlow row
// is vacuous for g>=0, R>=0, vlow<=vset -- checked on the host).
//
// Method (exact, terminates on KKT residuals; same algorithm and fixed point as the
// oracle's project_voltage): work on the dual
//     min_{lam>=0}  phi(lam) = 1/2 || [z - R lam]_+ ||^2 + u sum(lam)
// which is convex and piecewise quadratic, the pieces being the sets F of homes with g>0.
// Only a few tens of the ~10^3 voltage rows of a feeder ever carry a multiplier, so a column
// keeps a WORKING SET W of rows.  A launch of this kernel
//   1. reads the voltages  v = R g  of the stored iterate, produced for ALL rows and all
//      hours at once by the tensor-core contraction (contract_f64.cu),
//   2. drops rows whose multiplier is zero and admits the most violated rows (v > u),
//   3. iterates on W:  assemble the Hessian of the current piece  H = R_WF R_FW  (the only
//      step that streams rows of R, coalesced); minimise the piece EXACTLY over lam_W >= 0
//      with a primal-dual active-set loop that lives entirely in shared memory (blocked
//      Cholesky of H_AA, the sequential part inside one warp); search phi along the segment
//      to that minimiser.  If the active-set guesses cycle, take a projected-Newton arc step
//      with a Levenberg-Marquardt shift instead.
// Zones of up to 512 residences then recompute the voltages of ALL rows exactly for the new g
// (a warp per four rows) and go back to 2 inside the same launch; for larger zones the host
// alternates the launch with the screening contraction until no column has a violated row.
// The CTAs are persistent and pull columns from a per-class device queue.
//
// Three instantiations share the code (classes 1-3): |W| <= 32 (128 threads, ~30 KB of shared
// memory, 6 CTAs per SM), |W| <= 64 (256 threads, ~73 KB, 3 per SM) and |W| <= 128 (256
// threads, ~210 KB, 1 per SM); the first runs its active-set guesses in one warp (pdas_warp).
// Class 0 is the warp-per-column path of utility_qp_warp.cu for small columns.  A column carries a class flag; qp_init_kernel classifies it by the size
// of its warm-start set and a kernel hands it to the next class when it outgrows its own.
#include <algorithm>

#include <cuda_bf16.h>

#include "kernels.cuh"

namespace revs {

constexpr int kJT = 64;                  // columns of R per Hessian tile
constexpr int kTld = kJT + 1;
constexpr double kArcMin = 9.5367431640625e-07;   // 2^-20, shortest line-search step
constexpr int kChgMax = 128;             // most sign changes handled by a rank update of H
constexpr int kMaskWords = 512;          // feeders up to 16384 residences keep a mask of F
constexpr int kPdasMax = 40;             // active-set guesses per quadratic piece
constexpr double kHessShift = 1e-12;     // relative diagonal shift of the model Hessian

// Shared memory of one column.  Hb holds two things at once: the strict lower triangle of
// the model Hessian H (row i, column j<i at Hb[i*HLD+j], its diagonal in hdiag) and, in the
// unused upper part, the Cholesky factor of a principal sub-matrix, L(p,q) (p>=q) at
// Hb[q*HLD+p+1] -- so the active-set loop can refactor without reassembling H.
template <int WMAX, int THREADS>
struct QpSmem {
    double Hb[WMAX * (WMAX + 1)];
    double tileR[WMAX * kTld];
    double hdiag[WMAX];
    double lam[WMAX], trial[WMAX], grad[WMAX], dir[WMAX], b[WMAX], y[WMAX];
    double red[3 * (THREADS / 32)];
    double bcast[2];
    int idx[WMAX], fl[WMAX], inA[WMAX];
    int chg[kChgMax];                     // homes that changed side of g>0 (index*2 + left)
    unsigned fmask[kMaskWords];           // F the stored Hessian was formed for
    unsigned dmask[kMaskWords];           // scratch: homes that changed side since then
    unsigned short pairs[40];             // (p<<8 | q) of the lower-triangle pairs (small working sets)
    int ired[THREADS / 32];
    int ibcast[2];
};

// sum K values over the CTA with one barrier pair
template <int K, int THREADS, class S>
__device__ __forceinline__ void block_sum(double (&v)[K], S& sm) {
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = warp_sum(v[k]);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) sm.red[k * (THREADS / 32) + (threadIdx.x >> 5)] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double r = 0.0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) r += sm.red[k * (THREADS / 32) + w];
        v[k] = r;
    }
}
template <int THREADS, class S>
__device__ __forceinline__ double block_max(double v, S& sm) {
    v = warp_max(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm.red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = sm.red[0];
#pragma unroll
    for (int w = 1; w < THREADS / 32; ++w) r = fmax(r, sm.red[w]);
    return r;
}
template <int THREADS, class S>
__device__ __forceinline__ int block_count(bool p, S& sm) {
    const unsigned bal = __ballot_sync(0xffffffffu, p);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm.ired[threadIdx.x >> 5] = __popc(bal);
    __syncthreads();
    int r = 0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) r += sm.ired[w];
    return r;
}

// phi(lam) for multipliers lam[0..m) on rows idx[0..m); optionally stores g; optionally
// returns slope = sum grad_a (lam_a - base_a) in the same reduction.
template <int THREADS, class S>
__device__ double eval_phi(const double* __restrict__ R, int ld, int n, const double* __restrict__ z,
                           const int* idx, const double* lam, int m, double u, double* g_store, S& sm,
                           const double* grad = nullptr, const double* base = nullptr,
                           double* slope = nullptr, __nv_bfloat16* gbf_store = nullptr) {
    double acc[3] = {0.0, 0.0, 0.0};
    for (int j = threadIdx.x; j < n; j += THREADS) {
        double pi = 0.0;
        for (int a = 0; a < m; ++a) {
            const double l = lam[a];
            if (l != 0.0) pi = fma(R[(size_t)idx[a] * ld + j], l, pi);
        }
        const double gj = fmax(z[j] - pi, 0.0);
        if (g_store) {
            g_store[j] = gj;
            if (gbf_store) gbf_store[j] = __float2bfloat16_rn((float)gj);   // operand of the screening contraction
        }
        acc[0] = fma(gj, gj, acc[0]);
    }
    for (int a = threadIdx.x; a < m; a += THREADS) {
        acc[1] += lam[a];
        if (grad) acc[2] = fma(grad[a], lam[a] - base[a], acc[2]);
    }
    block_sum<3, THREADS>(acc, sm);
    if (slope) *slope = acc[2];
    return 0.5 * acc[0] + u * acc[1];
}

// Model Hessian H[p][q] = sum_{j in F} R[idx_p][j] R[idx_q][j] over the m working rows, F =
// homes with g>0 -> lower triangle of Hb and hdiag.  Threads form a 16 x (THREADS/16) grid;
// thread (tx,ty) owns rows ty + TY*a, columns tx + 16*b, a < NBP, b < NBQ; blocks that lie
// strictly above the diagonal are not computed.
//   INCR = false: from scratch, streaming all n columns of the working rows (coalesced).
//   INCR = true : rank-|list| correction  H += sum_c sgn_c r_c r_c^T  for the homes that
//                 entered (+) or left (-) F since H was last formed (chg list in smem).
// Either way sm.fmask ends up holding the bit mask of F the stored H corresponds to.
template <int WMAX, int THREADS, int NBP, int NBQ, bool INCR, class S>
__device__ void hessian(const double* __restrict__ R, int ld, int n, const double* g, int m, int nchg, S& sm) {
    constexpr int TY = THREADS / 16;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid & 15, ty = tid >> 4;
    double acc[NBP][NBQ];
#pragma unroll
    for (int a = 0; a < NBP; ++a)
#pragma unroll
        for (int b = 0; b < NBQ; ++b) acc[a][b] = 0.0;
    // the tile buffer holds kRows rows; fewer rows -> wider tiles -> fewer barriers
    constexpr int kRows = ((TY * NBP > 16 * NBQ) ? TY * NBP : 16 * NBQ) < WMAX ? ((TY * NBP > 16 * NBQ) ? TY * NBP : 16 * NBQ) : WMAX;
    constexpr int kJt = ((WMAX * kTld / kRows - 1) / 32 * 32) < 256 ? ((WMAX * kTld / kRows - 1) / 32 * 32) : 256;
    constexpr int kTl = kJt + 1;
    static_assert(kJt >= 32 && kRows * kTl <= WMAX * kTld, "tile does not fit");
    // rows beyond m read a zero row of the tile
    for (int p = m + warp; p < kRows; p += THREADS / 32)
        for (int l = lane; l < kJt; l += 32) sm.tileR[p * kTl + l] = 0.0;
    const int total = INCR ? nchg : n;
    for (int j0 = 0; j0 < total; j0 += kJt) {
        __syncthreads();
        for (int p = warp; p < m; p += THREADS / 32) {
            const double* row = R + (size_t)sm.idx[p] * ld;
#pragma unroll
            for (int l = lane; l < kJt; l += 32) {
                const int c = j0 + l;
                double val = 0.0;
                if (INCR) {
                    if (c < nchg) val = row[sm.chg[c] >> 1];
                } else {
                    if (c < n && g[c] > 0.0) val = row[c];
                }
                sm.tileR[p * kTl + l] = val;
            }
        }
        __syncthreads();
        const int jmax = min(kJt, total - j0);
#pragma unroll 4
        for (int jj = 0; jj < jmax; ++jj) {
            double pa[NBP], qb[NBQ];
            const double sg = INCR ? ((sm.chg[j0 + jj] & 1) ? -1.0 : 1.0) : 1.0;
#pragma unroll
            for (int a = 0; a < NBP; ++a) pa[a] = sm.tileR[(ty + TY * a) * kTl + jj] * sg;
#pragma unroll
            for (int b = 0; b < NBQ; ++b) qb[b] = sm.tileR[(tx + 16 * b) * kTl + jj];
#pragma unroll
            for (int a = 0; a < NBP; ++a)
#pragma unroll
                for (int b = 0; b < NBQ; ++b)
                    if (TY * (a + 1) > 16 * b) acc[a][b] = fma(pa[a], qb[b], acc[a][b]);
        }
    }
    __syncthreads();
#pragma unroll
    for (int a = 0; a < NBP; ++a)
#pragma unroll
        for (int b = 0; b < NBQ; ++b) {
            const int p = ty + TY * a, q = tx + 16 * b;
            if (p < m && q < m) {
                if (INCR) {
                    if (p > q) sm.Hb[p * (WMAX + 1) + q] += acc[a][b];
                    else if (p == q) sm.hdiag[p] += acc[a][b];
                } else {
                    if (p > q) sm.Hb[p * (WMAX + 1) + q] = acc[a][b];
                    else if (p == q) sm.hdiag[p] = acc[a][b];
                }
            }
        }
    __syncthreads();
}

// Small working sets (m <= kPairM): one (p,q) pair of the lower triangle per warp slot, the
// lanes split the columns, partial sums stay in registers over all tiles and are reduced
// with shuffles once at the end -- every thread does useful work and each accumulator is its
// own dependency chain.  Same contract as hessian<>.
constexpr int kPairM = 8;
constexpr int kPairMax = kPairM * (kPairM + 1) / 2;     // 36

template <int WMAX, int THREADS, bool INCR, class S>
__device__ void hessian_pairs(const double* __restrict__ R, int ld, int n, const double* g, int m, int nchg, S& sm) {
    constexpr int NW = THREADS / 32;
    constexpr int kAcc = (kPairMax + NW - 1) / NW;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int npairs = m * (m + 1) / 2;
    const int jt = min(256, (WMAX * kTld / m) & ~31), tl = jt + 1;
    double acc[kAcc];
#pragma unroll
    for (int k = 0; k < kAcc; ++k) acc[k] = 0.0;
    for (int idx = tid; idx < npairs; idx += THREADS) {   // pair index -> (p, q), p >= q
        int p = 0;
        while ((p + 1) * (p + 2) / 2 <= idx) ++p;
        sm.pairs[idx] = (unsigned short)((p << 8) | (idx - p * (p + 1) / 2));
    }
    const int total = INCR ? nchg : n;
    for (int j0 = 0; j0 < total; j0 += jt) {
        __syncthreads();
        for (int p = warp; p < m; p += NW) {
            const double* row = R + (size_t)sm.idx[p] * ld;
            for (int l = lane; l < jt; l += 32) {
                const int c = j0 + l;
                double val = 0.0;
                if (INCR) {
                    if (c < nchg) val = row[sm.chg[c] >> 1];
                } else if (c < n) {
                    const double rv = row[c];
                    val = g[c] > 0.0 ? rv : 0.0;
                }
                sm.tileR[p * tl + l] = val;
            }
        }
        __syncthreads();
        const int jmax = min(jt, total - j0);
#pragma unroll
        for (int k = 0; k < kAcc; ++k) {
            if (warp + k * NW >= npairs) break;
            const int pq = sm.pairs[warp + k * NW];
            const double* tp = sm.tileR + (pq >> 8) * tl;
            const double* tq = sm.tileR + (pq & 255) * tl;
            double a = acc[k];
            for (int l = lane; l < jmax; l += 32) {
                double prod = tp[l] * tq[l];
                if (INCR && (sm.chg[j0 + l] & 1)) prod = -prod;
                a += prod;
            }
            acc[k] = a;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kAcc; ++k) {
        if (warp + k * NW >= npairs) break;
        const double v = warp_sum(acc[k]);
        if (lane == 0) {
            const int pq = sm.pairs[warp + k * NW], p = pq >> 8, q = pq & 255;
            if (p == q) { if (INCR) sm.hdiag[p] += v; else sm.hdiag[p] = v; }
            else { double* h = &sm.Hb[p * (WMAX + 1) + q]; if (INCR) *h += v; else *h = v; }
        }
    }
    __syncthreads();
}

// Compare F = {g>0} with the mask the stored H was formed for.  Returns the number of homes
// that changed side (index*2 + left? in sm.chg, ascending), or -1 if there are more than
// kChgMax (the caller then recomputes H from scratch).  Updates the mask.  Every warp owns a
// contiguous range of 32-home words, so ordering needs one prefix over the warps only.
template <int THREADS, class S>
__device__ int mask_changes(const double* g, int n, S& sm) {
    constexpr int NW = THREADS / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwords = (n + 31) >> 5, wpw = (nwords + NW - 1) / NW;
    const int w0 = warp * wpw, w1 = min(nwords, w0 + wpw);
    int cnt = 0;
    for (int w = w0; w < w1; ++w) {
        const int j = (w << 5) + lane;
        const unsigned now = __ballot_sync(0xffffffffu, j < n && g[j] > 0.0);
        const unsigned diff = now ^ sm.fmask[w];
        if (lane == 0) { sm.fmask[w] = now; sm.dmask[w] = diff; }
        cnt += __popc(diff);
    }
    if (lane == 0) sm.ired[warp] = cnt;
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        before += (w < warp) ? sm.ired[w] : 0;
        total += sm.ired[w];
    }
    if (total <= kChgMax) {
        int pos = before;
        for (int w = w0; w < w1; ++w) {
            const unsigned diff = sm.dmask[w], now = sm.fmask[w];
            if ((diff >> lane) & 1u)
                sm.chg[pos + __popc(diff & ((1u << lane) - 1))] = ((((w << 5) + lane)) << 1) | (((now >> lane) & 1u) ? 0 : 1);
            pos += __popc(diff);
        }
    }
    __syncthreads();
    return total > kChgMax ? -1 : total;
}

// ---- dense SPD solves in shared memory on a principal sub-matrix of H.  The factor lives
// in the upper part of Hb: L(p,q) = Hb[q*HLD + p + 1].  Blocked by 32 so that the
// sequential part runs inside one warp (lanes own rows, __syncwarp / shuffles only) and the
// CTA meets at three barriers per 32 columns instead of three per column.
#define LV(p, q) Hb[(q) * HLD + (p) + 1]

// Factor H[fl,fl] + shift*I (fl ascending, ma entries) and solve for rhs y[0..ma) in place.
template <int WMAX, int THREADS, class S>
__device__ void factor_solve(int ma, double shift, S& sm) {
    constexpr int HLD = WMAX + 1;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* Hb = sm.Hb;
    double* y = sm.y;
    // gather the sub-matrix into the factor storage
    for (int e = tid; e < ma * ma; e += THREADS) {
        const int p = e % ma, q = e / ma;
        if (p < q) continue;
        const int ip = sm.fl[p], iq = sm.fl[q];
        LV(p, q) = (p == q) ? sm.hdiag[ip] + shift : Hb[ip * HLD + iq];
    }
    __syncthreads();
    for (int kb = 0; kb < ma; kb += 32) {
        const int bs = min(32, ma - kb), r0 = kb + bs, rem = ma - r0;
        if (warp == 0) {                                   // diagonal block, lanes own rows
            const bool row = lane < bs;
            for (int k = 0; k < bs; ++k) {
                const double dkk = sqrt(fmax(LV(kb + k, kb + k), 1e-300));
                __syncwarp();
                if (lane == k) LV(kb + k, kb + k) = dkk;
                double lik = 0.0;
                if (row && lane > k) { lik = LV(kb + lane, kb + k) / dkk; LV(kb + lane, kb + k) = lik; }
                __syncwarp();
                if (row && lane > k)
                    for (int j = k + 1; j <= lane; ++j)
                        LV(kb + lane, kb + j) = fma(-lik, LV(kb + j, kb + k), LV(kb + lane, kb + j));
                __syncwarp();
            }
        }
        __syncthreads();
        if (rem > 0) {
            for (int r = tid; r < rem; r += THREADS) {     // panel below the block, one thread per row
                const int i = r0 + r;
                for (int k = 0; k < bs; ++k) {
                    double acc = LV(i, kb + k);
                    for (int q = 0; q < k; ++q) acc = fma(-LV(i, kb + q), LV(kb + k, kb + q), acc);
                    LV(i, kb + k) = acc / LV(kb + k, kb + k);
                }
            }
            __syncthreads();
            for (int e = tid; e < rem * rem; e += THREADS) {   // trailing lower triangle
                const int i = e % rem, j = e / rem;
                if (j > i) continue;
                double acc = 0.0;
                for (int k = 0; k < bs; ++k) acc = fma(LV(r0 + i, kb + k), LV(r0 + j, kb + k), acc);
                LV(r0 + i, r0 + j) -= acc;
            }
            __syncthreads();
        }
    }
    for (int kb = 0; kb < ma; kb += 32) {                  // L y = b
        const int bs = min(32, ma - kb), r0 = kb + bs;
        if (warp == 0) {
            double v = lane < bs ? y[kb + lane] : 0.0;
            for (int k = 0; k < bs; ++k) {
                const double yk = __shfl_sync(0xffffffffu, v, k) / LV(kb + k, kb + k);
                if (lane == k) v = yk;
                if (lane > k && lane < bs) v = fma(-LV(kb + lane, kb + k), yk, v);
            }
            if (lane < bs) y[kb + lane] = v;
        }
        __syncthreads();
        for (int i = r0 + tid; i < ma; i += THREADS) {
            double acc = y[i];
            for (int k = 0; k < bs; ++k) acc = fma(-LV(i, kb + k), y[kb + k], acc);
            y[i] = acc;
        }
        __syncthreads();
    }
    for (int kb = ((ma - 1) / 32) * 32; kb >= 0; kb -= 32) {   // L^T x = y
        const int bs = min(32, ma - kb);
        if (warp == 0) {
            double v = lane < bs ? y[kb + lane] : 0.0;
            for (int k = bs - 1; k >= 0; --k) {
                const double xk = __shfl_sync(0xffffffffu, v, k) / LV(kb + k, kb + k);
                if (lane == k) v = xk;
                if (lane < k) v = fma(-LV(kb + k, kb + lane), xk, v);
            }
            if (lane < bs) y[kb + lane] = v;
        }
        __syncthreads();
        for (int i = tid; i < kb; i += THREADS) {
            double acc = y[i];
            for (int k = 0; k < bs; ++k) acc = fma(-LV(kb + k, i), y[kb + k], acc);
            y[i] = acc;
        }
        __syncthreads();
    }
}
#undef LV

// ordered list fl[0..) of the rows i < m with flag[i] != 0; returns its length
template <int THREADS, class S>
__device__ int compact_flags(const int* flag, int m, S& sm) {
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        int base = 0;
        for (int i0 = 0; i0 < m; i0 += 32) {
            const int i = i0 + lane;
            const bool on = i < m && flag[i] != 0;
            const unsigned bal = __ballot_sync(0xffffffffu, on);
            if (on) sm.fl[base + __popc(bal & ((1u << lane) - 1))] = i;
            base += __popc(bal);
        }
        if (lane == 0) sm.ibcast[1] = base;
    }
    __syncthreads();
    return sm.ibcast[1];
}

// (H v)_i over the m working rows for a vector v supported on fl[0..ma): thread per row
template <int WMAX, class S>
__device__ __forceinline__ double hess_row_dot(int i, const double* v, int ma, S& sm) {
    constexpr int HLD = WMAX + 1;
    double acc = 0.0;
    for (int p = 0; p < ma; ++p) {
        const int j = sm.fl[p];
        const double h = (i > j) ? sm.Hb[i * HLD + j] : ((i < j) ? sm.Hb[j * HLD + i] : sm.hdiag[i]);
        acc = fma(h, v[j], acc);
    }
    return acc;
}

// Primal-dual active-set minimisation of one quadratic piece for working sets of up to 32 rows,
// executed by ONE warp (lanes = rows) without block barriers: the first CTA class spends most of
// its time here and the block-wide version costs a dozen __syncthreads per guess.  Same
// arithmetic as the block version below: b = H lam + shift lam - grad, A = {lam > 0} u {grad < 0},
// solve (H_AA + shift I) x_A = b_A, flip the rows with x <= 0 (in A) or mu < 0 (outside).
// Returns whether the guesses settled; the minimiser is left in sm.trial.
template <int WMAX, class S>
__device__ bool pdas_warp(int m, double shift, S& sm, unsigned& n_pdas, double& flops) {
    constexpr int HLD = WMAX + 1;
    double* Hb = sm.Hb;
#define LVW(p, q) Hb[(q) * HLD + (p) + 1]
    const int lane = threadIdx.x & 31;
    const unsigned full = 0xffffffffu;
    const bool row = lane < m;
    auto Hij = [&](int i, int j) -> double { return i > j ? Hb[i * HLD + j] : (i < j ? Hb[j * HLD + i] : sm.hdiag[i]); };
    const double lam = row ? sm.lam[lane] : 0.0, grad = row ? sm.grad[lane] : 0.0;
    double b = 0.0;
    for (int q = 0; q < m; ++q) {
        const double lq = __shfl_sync(full, lam, q);
        if (row && lq > 0.0) b = fma(Hij(lane, q), lq, b);
    }
    b += shift * lam - grad;
    bool inA = row && (lam > 0.0 || grad < 0.0);
    double x = 0.0;
    bool settled = false;
    for (int guess = 0; guess < kPdasMax; ++guess) {
        ++n_pdas;
        const unsigned Am = __ballot_sync(full, inA);
        const int ma = __popc(Am);
        const int pos = __popc(Am & ((1u << lane) - 1));
        flops += (2.0 / 3.0) * ma * ma * ma + 4.0 * ma * ma + 2.0 * m * ma;
        double xs = 0.0;
        if (ma > 0) {
            const int o = lane < ma ? (int)__fns(Am, 0, lane + 1) : 0;       // original row of compact row `lane`
            for (int c = 0; c < ma; ++c) {
                const int oc = __shfl_sync(full, o, c);
                if (lane < ma && c <= lane) LVW(lane, c) = Hij(o, oc) + (c == lane ? shift : 0.0);
            }
            __syncwarp();
            double rdiag = 1.0;
            for (int k = 0; k < ma; ++k) {                                    // Cholesky, left-looking, lanes own rows
                double sv = 0.0;
                if (lane >= k && lane < ma) {
                    sv = LVW(lane, k);
                    for (int p = 0; p < k; ++p) sv = fma(-LVW(lane, p), LVW(k, p), sv);
                }
                const double skk = fmax(__shfl_sync(full, sv, k), 1e-300);
                const double rk = rsqrt(skk);                                 // instead of sqrt + divide
                const double dkk = skk * rk;
                if (lane == k) rdiag = rk;                                    // reciprocal pivots in registers
                if (lane >= k && lane < ma) LVW(lane, k) = lane == k ? dkk : sv * rk;
                __syncwarp();
            }
            double y = __shfl_sync(full, b, o);                               // rhs of compact row `lane`
            if (lane >= ma) y = 0.0;
            for (int k = 0; k < ma; ++k) {
                const double yk = __shfl_sync(full, y, k) * __shfl_sync(full, rdiag, k);
                if (lane == k) y = yk;
                if (lane > k && lane < ma) y = fma(-LVW(lane, k), yk, y);
            }
            for (int k = ma - 1; k >= 0; --k) {
                const double xk = __shfl_sync(full, y, k) * __shfl_sync(full, rdiag, k);
                if (lane == k) y = xk;
                if (lane < k) y = fma(-LVW(k, lane), xk, y);
            }
            xs = y;
        }
        const double xg = __shfl_sync(full, xs, pos & 31);
        x = inA ? xg : 0.0;
        double mu = 0.0;
        for (int q = 0; q < m; ++q) {
            const double xq = __shfl_sync(full, x, q);
            if (row && xq != 0.0) mu = fma(Hij(lane, q), xq, mu);
        }
        mu -= b;
        const bool bad = row && (inA ? (x <= 0.0) : (mu < 0.0));
        if (!__any_sync(full, bad)) { settled = true; break; }
        if (bad) inA = !inA;
        __syncwarp();
    }
    if (row) sm.trial[lane] = x;
#undef LVW
    return settled;
}

constexpr int kAddMaxVerify = 8;
constexpr int kCtaPassMax = 16;          // admit / solve / verify passes of one launch (zones <= kVerifyMaxN)

// exact voltages of ALL rows for the g in global memory: one warp per row
template <int THREADS>
__device__ void exact_voltages(const double* __restrict__ R, int ld, int n, const double* g, double* v) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int NW = THREADS / 32;
    for (int i0 = 4 * warp; i0 < n; i0 += 4 * NW) {       // four rows per warp step: loads and reductions overlap
        double a[4] = {0.0, 0.0, 0.0, 0.0};
        for (int k = lane; k < n; k += 32) {
            const double gk = g[k];
#pragma unroll
            for (int q = 0; q < 4; ++q) a[q] = fma(R[(size_t)min(i0 + q, n - 1) * ld + k], gk, a[q]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int q = 0; q < 4; ++q) a[q] += __shfl_xor_sync(0xffffffffu, a[q], o);
        }
        if (lane < 4 && i0 + lane < n) v[i0 + lane] = lane == 0 ? a[0] : (lane == 1 ? a[1] : (lane == 2 ? a[2] : a[3]));
    }
    __syncthreads();
}

template <int WMAX, int THREADS, int CLS, class S>
__device__ void qp_column(const QpParams& P, const int c, S& sm) {
    constexpr bool BIG = CLS == kQpClasses - 1;   // last class: nowhere to hand a column on to
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int f = c / P.T, t = c % P.T;
    long long tr_start = 0;
    const long long tr_clk0 = clock64();
    if (P.trace) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_start));
    if (P.status[c] != 0) return;
    if (P.cls[c] != CLS) return;   // column of another instantiation

    const FeederDev fd = P.feeders[f];
    const int n = fd.n, ld = fd.np;
    const double* R = P.Rpool + fd.roff;
    const size_t col = (size_t)t * P.Hp + fd.off;
    const double* z = P.z_t + col;
    double* lam_g = P.lam_t + col;
    double* g = P.g_t + col;
    double* v = P.v_t + col;
    const double u = P.u, tol = P.tol;
    const double* rn2 = P.rn2 + fd.off;
    int* widx = P.widx + (size_t)c * kWMax;

    // Zones up to kVerifyMaxN residences finish inside this launch: after the restricted solve
    // the voltages of ALL rows are recomputed exactly for the new g (a warp per row, the block
    // of R is L2-resident) and violated rows are admitted in a further pass.  Larger zones leave
    // the check to the next tensor-core screening pass of the host loop.
    const bool self_verify = n <= kVerifyMaxN;
    int inner_prev = P.inner_ok[c];   // 1 solved earlier; 2/3 handed over in this round (3: g changed since the screen)
    unsigned long long its_all = 0;
    unsigned n_evals = 0, n_pdas = 0, n_fallback = 0;
    double flops = 0.0;
    long long tc[5] = {0, 0, 0, 0, 0}, t0 = clock64(), t1;   // phase cycles (debug)
    int m = 0, ok = 0;
    bool finished = false, handed = false;
    for (int pass = 0; pass < kCtaPassMax; ++pass) {
    // ------------------------------------------------------------ working set
    bool clean = false;   // no violated row found: v is still valid if g stays put
    {
        if (pass == 0 && P.sweep && inner_prev == 3 && self_verify) {
            exact_voltages<THREADS>(R, ld, n, g, v);
        } else if (P.v32_t && pass == 0) {
            // Voltages came from the BF16 screening pass: rows at or below (1-margin) u are
            // proven feasible; every other row without a multiplier is a candidate whose
            // voltage is recomputed here exactly (FP64 row of R times g), one warp per row.
            const float* v32 = P.v32_t + col;
            const double thr = (1.0 - kScreenMargin) * u;
            for (int j0 = 0; j0 < n; j0 += THREADS) {
                const int j = j0 + tid;
                const float a = j < n ? v32[j] : 0.f;
                const bool cand = j < n && (double)a > thr && !(lam_g[j] > 0.0);
                if (j < n && !cand) v[j] = (double)a;
                unsigned bal = __ballot_sync(0xffffffffu, cand);
                while (bal) {
                    const int bit = __ffs(bal) - 1;
                    bal &= bal - 1;
                    const int row_i = j0 + warp * 32 + bit;
                    const double* row = R + (size_t)row_i * ld;
                    double acc = 0.0;
                    for (int k = lane; k < n; k += 32) acc = fma(row[k], g[k], acc);
                    acc = warp_sum(acc);
                    if (lane == 0) v[row_i] = acc;
                }
            }
            __syncthreads();
        }
        const int m_old = P.wcount[c];
        // keep rows with a positive multiplier (serial compaction keeps the order stable)
        if (tid == 0) {
            int k = 0;
            for (int a = 0; a < m_old; ++a) {
                int i = widx[a];
                double l = lam_g[i];
                if (l > 0.0) { sm.idx[k] = i; sm.lam[k] = l; ++k; }
            }
            sm.ibcast[0] = k;
        }
        __syncthreads();
        m = sm.ibcast[0];
        // violated rows outside W, most violated first; key order (viol desc, index asc)
        double prev_v = 1e300;
        int prev_i = -1;
        int added = 0, n_viol_left = 0;
        // zones that verify in-kernel admit few rows per pass: after a re-solve with the most violated
        // rows most neighbouring violations are gone
        const int room = min(self_verify ? kAddMaxVerify : kAddMax, WMAX - m);
        for (int round = 0; round <= room; ++round) {
            double best = -1.0;
            int besti = 0x7fffffff;
            for (int j = tid; j < n; j += THREADS) {
                const double viol = v[j] - u;
                if (viol > tol && !(lam_g[j] > 0.0)) {
                    bool after_prev = (viol < prev_v) || (viol == prev_v && j > prev_i);
                    if (after_prev && (viol > best || (viol == best && j < besti))) { best = viol; besti = j; }
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                double ob = __shfl_xor_sync(0xffffffffu, best, o);
                int oi = __shfl_xor_sync(0xffffffffu, besti, o);
                if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
            }
            __syncthreads();
            if (lane == 0) { sm.red[warp] = best; sm.ired[warp] = besti; }
            __syncthreads();
            best = sm.red[0]; besti = sm.ired[0];
#pragma unroll
            for (int w = 1; w < THREADS / 32; ++w) {
                if (sm.red[w] > best || (sm.red[w] == best && sm.ired[w] < besti)) { best = sm.red[w]; besti = sm.ired[w]; }
            }
            if (best < 0.0) break;              // no further violated row
            if (round == room) { n_viol_left = 1; break; }
            if (tid == 0) { sm.idx[m + added] = besti; sm.lam[m + added] = 0.0; }
            ++added;
            prev_v = best; prev_i = besti;
        }
        __syncthreads();
        if (added == 0 && n_viol_left == 0 && inner_prev == 1) {
            if (tid == 0) P.status[c] = 1;      // KKT point of the full problem
            finished = true;
            break;
        }
        if (n_viol_left && m + added == WMAX) {
            if (!BIG) {                         // hand the column over (state consistent; 3: g moved since the screen)
                if (tid == 0) {
                    P.cls[c] = CLS + 1;
                    P.inner_ok[c] = (pass > 0 || inner_prev == 3) ? 3 : 2;
                    atomicAdd(P.n_running, 1);
                    atomicAdd(P.n_cls + CLS + 1, 1);
                }
                handed = true;
                break;
            }
            // a full working set overflows only once it has been solved: rows of a warm start that was never solved
            // on W may leave it with a zero multiplier (solve first, admit in the next pass)
            if (added == 0 && inner_prev == 1) {
                if (tid == 0) { P.status[c] = 2; atomicAdd(P.n_failed, 1); }
                finished = true;
                break;
            }
        }
        clean = (added == 0 && n_viol_left == 0);
        // clear the stored multipliers of the old set; rewritten at the end
        for (int a = tid; a < m_old; a += THREADS) lam_g[widx[a]] = 0.0;
        m += added;
        __syncthreads();
    }

    // ------------------------------------------------------------ piecewise-quadratic descent on W
    __nv_bfloat16* gbf = P.gbf_t ? reinterpret_cast<__nv_bfloat16*>(P.gbf_t) + col : nullptr;
    double phi = eval_phi<THREADS>(R, ld, n, z, sm.idx, sm.lam, m, u, g, sm, nullptr, nullptr, nullptr, gbf);
    double tau = 1.0;
    int its = 0;
    ok = 0;
    flops += 2.0 * m * n;                       // algorithmic FP64 flops of this launch (first evaluation)
    bool have_H = false;   // Hb/hdiag hold the Hessian for the mask in sm.fmask
#define PHASE(i) do { t1 = clock64(); tc[i] += t1 - t0; t0 = t1; } while (0)
    const int inner_max = P.inner_max;
    double scale = 0.0;                         // mean |R_a|^2 over W: curvature scale of the Hessian shifts
    if (inner_max > 0 && m > 0) {
        double sc[1] = {0.0};
        for (int a = tid; a < m; a += THREADS) sc[0] += rn2[sm.idx[a]];
        block_sum<1, THREADS>(sc, sm);
        scale = sc[0] / (double)m;
    }
    for (; its < inner_max; ++its) {
        __syncthreads();
        // gradient on W:  u - R[idx_a] . g
        for (int a = warp; a < m; a += THREADS / 32) {
            const double* row = R + (size_t)sm.idx[a] * ld;
            double acc = 0.0;
            for (int j = lane; j < n; j += 32) acc = fma(row[j], g[j], acc);
            acc = warp_sum(acc);
            if (lane == 0) sm.grad[a] = u - acc;
        }
        __syncthreads();
        double kk = 0.0;
        for (int a = tid; a < m; a += THREADS) {
            double gr = sm.grad[a];
            kk = fmax(kk, fabs(sm.lam[a] > 0.0 ? gr : fmin(gr, 0.0)));
        }
        const double kkt = block_max<THREADS>(kk, sm);
        PHASE(0);
        flops += 2.0 * m * n;
        if (kkt < tol) { ok = 1; break; }

        // model Hessian of the current piece on all of W (register block sized to m): from
        // scratch on the first piece of a launch, afterwards a rank update for the few homes
        // that crossed g = 0
        {
            int nchg = -1;
            if (n <= kMaskWords * 32) {
                if (have_H) nchg = mask_changes<THREADS>(g, n, sm);
                else {
                    for (int w = tid; w < (n + 31) / 32; w += THREADS) sm.fmask[w] = 0u;
                    __syncthreads();
                    (void)mask_changes<THREADS>(g, n, sm);       // records F; H is formed below
                }
            }
            constexpr int TY = THREADS / 16;
            const int nq = (m + 15) >> 4, np_ = (m + TY - 1) / TY;
            (void)nq; (void)np_;
            if (m <= kPairM) {
                if (have_H && nchg >= 0) { if (nchg > 0) hessian_pairs<WMAX, THREADS, true>(R, ld, n, g, m, nchg, sm); }
                else hessian_pairs<WMAX, THREADS, false>(R, ld, n, g, m, 0, sm);
            } else {
#define HESS(NP, NQ)                                                                          \
    do {                                                                                      \
        if (have_H && nchg >= 0) { if (nchg > 0) hessian<WMAX, THREADS, NP, NQ, true>(R, ld, n, g, m, nchg, sm); } \
        else hessian<WMAX, THREADS, NP, NQ, false>(R, ld, n, g, m, 0, sm);                     \
    } while (0)
            if constexpr (WMAX == 32) {            // TY = 8: rows in blocks of 8, columns of 16
                if (np_ <= 1) HESS(1, 1);
                else if (np_ <= 2) HESS(2, 1);
                else if (np_ <= 3) HESS(3, 2);
                else HESS(4, 2);
            } else {                               // TY = 16
                if (nq <= 1) HESS(1, 1);
                else if (nq <= 2) HESS(2, 2);
                else if (nq <= 3) HESS(3, 3);
                else if (nq <= 4 || WMAX == 64) HESS(4, 4);
                else if (nq <= 6) HESS((WMAX > 64 ? 6 : 4), (WMAX > 64 ? 6 : 4));
                else HESS((WMAX > 64 ? 8 : 4), (WMAX > 64 ? 8 : 4));
            }
#undef HESS
            }
            flops += (double)m * (m + 1) * ((nchg >= 0 && have_H) ? nchg : n);   // lower triangle, 2 flops per MAC
            have_H = true;
        }
        PHASE(1);
        const double shift = kHessShift * scale + 1e-300;

        // ---- exact minimiser of the piece over lam_W >= 0: primal-dual active set
        // b = H lam - grad ; A = {lam > 0} u {grad < 0}
        bool pdas_ok = false;
        if constexpr (WMAX <= 32) {
            __syncthreads();
            if (warp == 0) {
                const bool settled = pdas_warp<WMAX>(m, shift, sm, n_pdas, flops);
                if (lane == 0) sm.ibcast[1] = settled ? 1 : 0;
            }
            __syncthreads();
            pdas_ok = sm.ibcast[1] != 0;
        } else {
            for (int a = tid; a < m; a += THREADS) sm.inA[a] = (sm.lam[a] > 0.0) ? 1 : 0;
            __syncthreads();
            int ma = compact_flags<THREADS>(sm.inA, m, sm);
            for (int i = tid; i < m; i += THREADS)
                sm.b[i] = hess_row_dot<WMAX>(i, sm.lam, ma, sm) + shift * sm.lam[i] - sm.grad[i];
            __syncthreads();
            for (int a = tid; a < m; a += THREADS) sm.inA[a] = (sm.lam[a] > 0.0 || sm.grad[a] < 0.0) ? 1 : 0;
            __syncthreads();
            for (int guess = 0; guess < kPdasMax; ++guess) {
                ++n_pdas;
                ma = compact_flags<THREADS>(sm.inA, m, sm);
                flops += (2.0 / 3.0) * ma * ma * ma + 4.0 * ma * ma + 2.0 * m * ma;
                for (int a = tid; a < m; a += THREADS) sm.trial[a] = 0.0;
                if (ma > 0) {
                    for (int p = tid; p < ma; p += THREADS) sm.y[p] = sm.b[sm.fl[p]];
                    __syncthreads();
                    factor_solve<WMAX, THREADS>(ma, shift, sm);
                    for (int p = tid; p < ma; p += THREADS) sm.trial[sm.fl[p]] = sm.y[p];
                }
                __syncthreads();
                bool bad = false;
                for (int i = tid; i < m; i += THREADS) {
                    if (sm.inA[i]) {
                        if (sm.trial[i] <= 0.0) { bad = true; sm.inA[i] = 0; }
                    } else {
                        const double mu = hess_row_dot<WMAX>(i, sm.trial, ma, sm) - sm.b[i];
                        if (mu < 0.0) { bad = true; sm.inA[i] = 1; }
                    }
                }
                if (block_count<THREADS>(bad, sm) == 0) { pdas_ok = true; break; }
            }

        }

        PHASE(2);
        double alpha = 1.0, phin = phi;
        bool stepped = false;
        if (pdas_ok) {
            // search phi on the segment lam -> minimiser (both feasible)
            for (int a = tid; a < m; a += THREADS) sm.dir[a] = sm.trial[a] - sm.lam[a];
            __syncthreads();
            for (alpha = 1.0; alpha >= kArcMin; alpha *= 0.5) {
                for (int a = tid; a < m; a += THREADS) sm.trial[a] = fmax(fma(alpha, sm.dir[a], sm.lam[a]), 0.0);
                __syncthreads();
                double slope;
                phin = eval_phi<THREADS>(R, ld, n, z, sm.idx, sm.trial, m, u, nullptr, sm, sm.grad, sm.lam, &slope);
                ++n_evals;
                flops += 2.0 * m * n;
                // + rounding noise of phi itself, see oracle/revs_oracle.py:project_voltage
                if (phin <= phi + 1e-4 * slope + 1e-14 * fabs(phi)) { stepped = true; break; }
            }
        }
        if (!stepped) {
            // safeguard: projected-Newton arc step on the free rows with an LM shift
            ++n_fallback;
            const double eps = fmin(1e-8, kkt);
            for (int a = tid; a < m; a += THREADS) {
                const bool bound = (sm.lam[a] <= eps) && (sm.grad[a] > 0.0);
                sm.inA[a] = bound ? 0 : 1;
            }
            __syncthreads();
            const int mf = compact_flags<THREADS>(sm.inA, m, sm);
            for (;;) {
                for (int a = tid; a < m; a += THREADS) sm.dir[a] = -sm.lam[a];
                if (mf > 0) {
                    for (int p = tid; p < mf; p += THREADS) sm.y[p] = -sm.grad[sm.fl[p]];
                    __syncthreads();
                    factor_solve<WMAX, THREADS>(mf, 1e-10 * tau * scale + 1e-300, sm);
                    for (int p = tid; p < mf; p += THREADS) sm.dir[sm.fl[p]] = sm.y[p];
                }
                __syncthreads();
                bool found = false;
                for (alpha = 1.0; alpha >= kArcMin; alpha *= 0.5) {
                    for (int a = tid; a < m; a += THREADS) sm.trial[a] = fmax(fma(alpha, sm.dir[a], sm.lam[a]), 0.0);
                    __syncthreads();
                    double slope;
                    phin = eval_phi<THREADS>(R, ld, n, z, sm.idx, sm.trial, m, u, nullptr, sm, sm.grad, sm.lam, &slope);
                    ++n_evals;
                    flops += 2.0 * m * n;
                    if (phin <= phi + 1e-4 * slope + 1e-14 * fabs(phi)) { found = true; break; }
                }
                if (found || tau > 1e40 || mf == 0) break;
                tau *= 1e3;
            }
            if (alpha == 1.0) tau = fmax(1.0, tau / 10.0);
        }
        PHASE(3);
        __syncthreads();
        for (int a = tid; a < m; a += THREADS) sm.lam[a] = sm.trial[a];
        __syncthreads();
        phi = eval_phi<THREADS>(R, ld, n, z, sm.idx, sm.lam, m, u, g, sm, nullptr, nullptr, nullptr, gbf);
        flops += 2.0 * m * n;
        PHASE(4);
    }

    // ------------------------------------------------------------ persist
    __syncthreads();
    for (int a = tid; a < m; a += THREADS) {
        lam_g[sm.idx[a]] = sm.lam[a];
        widx[a] = sm.idx[a];
    }
    // no violated row and the stored iterate already satisfies KKT on W: it is the solution
    // (g was not touched, so the voltages the violation scan used are its voltages)
    const bool done = clean && ok && its == 0;
    its_all += (unsigned long long)its;
    if (tid == 0) {
        P.wcount[c] = m;
        P.inner_ok[c] = ok;
        P.status[c] = done ? 1 : 0;
    }
    if (done) { finished = true; break; }
    if (!self_verify || !ok || inner_max <= 0) break;      // the next screening pass checks the other rows
    __syncthreads();
    exact_voltages<THREADS>(R, ld, n, g, v);
    flops += 2.0 * n * n;
    inner_prev = 1;
    }   // pass

    if (tid == 0) {
        if (!finished && !handed) { atomicAdd(P.n_running, 1); atomicAdd(P.n_cls + CLS, 1); }
        atomicAdd(P.newton_its, its_all);
        atomicAdd(P.cols, 1ull);
        atomicMax(P.max_ws, m);
        atomicAdd(P.flops, (unsigned long long)flops);
        const unsigned long long its = its_all;
        if (P.trace) {
            long long tr_end; unsigned smid;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_end));
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            long long* rec = P.trace + 12 * (size_t)c;
            rec[0] = tr_start; rec[1] = tr_end; rec[2] = smid; rec[3] = ((long long)CLS << 40) | ((long long)m << 20) | its;
            for (int i = 0; i < 5; ++i) rec[4 + i] = tc[i];
            rec[9] = n_pdas; rec[10] = n_evals; rec[11] = clock64() - tr_clk0;
        }
        if (P.dbg) {
            atomicAdd(P.dbg + 0, (unsigned long long)n_evals);
            atomicAdd(P.dbg + 1, (unsigned long long)n_pdas);
            atomicMax(P.dbg + 2, (unsigned long long)its);
            atomicAdd(P.dbg + 3, (unsigned long long)n_fallback);
            for (int i = 0; i < 5; ++i) atomicAdd(P.dbg + 4 + 5 * CLS + i, (unsigned long long)tc[i]);
        }
    }
}

// The kernel proper: CTAs pull the running columns of their class from a device-side queue
// (list built by order_columns_kernel), so the grid does not depend on counts the host would
// have to read back.
template <int WMAX, int THREADS, int CLS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) utility_qp_kernel(QpParams P) {
    using S = QpSmem<WMAX, THREADS>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    S& sm = *reinterpret_cast<S*>(smem_raw);
    const int count = P.order_count[CLS];
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) sm.ibcast[0] = atomicAdd(P.queue + CLS, 1);
        __syncthreads();
        const int slot = sm.ibcast[0];
        if (slot >= count) break;
        qp_column<WMAX, THREADS, CLS>(P, P.order[(size_t)CLS * P.ncols + slot], sm);
    }
}

// Work lists for one working-set round (block-level counts, one atomic per list and CTA):
// lists 1..3 = running columns of the CTA classes, lists 4..7 = the warp kernel's columns by
// working-set size (>= 3, 2, 1, 0).  mode 0 (first round): a warp-class column without
// multipliers and without a screening candidate is already solved (g = [z]_+) and never
// reaches a QP kernel.  mode 2 (sweep): only columns handed over during this round.
// order_count must be zero.  mode < 0: mode 0 / 1 by the device round counter.
__global__ void __launch_bounds__(256) order_columns_kernel(QpParams P, int mode, int* __restrict__ order,
                                                            int* __restrict__ order_count) {
    __shared__ int cnt[kQpLists], base[kQpLists];
    const int tid = threadIdx.x;
    if (tid < kQpLists) cnt[tid] = 0;
    __syncthreads();
    const int c = blockIdx.x * blockDim.x + tid;
    int li = -1, pos = 0;
    FeederDev fd{};
    if (mode < 0) mode = (P.round_ctr && *P.round_ctr > 0) ? 1 : 0;     // captured graph: the round counter lives on the device
    if (c < P.ncols && P.status[c] == 0) {
        const int cl = P.cls[c];
        if (mode == 2) {
            if (cl >= 1 && P.inner_ok[c] >= 2) li = cl;
        } else if (cl >= 1) {
            li = cl;
        } else {
            const int m = P.wcount[c];
            if (mode == 0 && m == 0 && P.cand && P.cand[c] == 0) { P.status[c] = 1; P.inner_ok[c] = 1; }
            else {
                fd = P.feeders[c / P.T];
                li = (fd.n <= 128 ? kQpClasses : (fd.n <= 256 ? kQpClasses + kQpBuckets : kListBig)) + (m >= 3 ? 0 : 3 - m);
            }
        }
        if (li >= 0) pos = atomicAdd(&cnt[li], 1);
    }
    __syncthreads();
    if (tid < kQpLists) base[tid] = cnt[tid] ? atomicAdd(&order_count[tid], cnt[tid]) : 0;
    __syncthreads();
    if (li >= kQpClasses)       // warp kernels: everything a column needs to start loading, in one 16-byte entry
        P.order4[(size_t)(li - kQpClasses) * P.ncols + base[li] + pos] =
            make_int4(c, (int)fd.off, fd.n | (fd.np << 16), (int)(fd.roff >> 4));
    else if (li >= 0) order[(size_t)li * P.ncols + base[li] + pos] = c;
}

cudaError_t launch_order_columns(const QpParams& P, int mode, int* order, int* order_count, cudaStream_t stream) {
    cudaError_t e = cudaMemsetAsync(order_count, 0, 2 * kQpLists * sizeof(int), stream);   // counts and queue heads
    if (e != cudaSuccess) return e;
    order_columns_kernel<<<(P.ncols + 255) / 256, 256, 0, stream>>>(P, mode, order, order_count);
    return cudaGetLastError();
}

__global__ void round_end_kernel(RoundEndParams P) {
    if (threadIdx.x != 0) return;
    const int running = *P.n_running;
    const int round = *P.round_ctr + 1;
    *P.round_ctr = round;
    *P.rounds_total += 1ull;
    const bool err = *P.n_failed != 0 || *P.infeasible != 0;
    bool more = running > 0 && !err;
    if (more && round >= P.round_max) { *P.noconv = 1; more = false; }
    if (P.use_cond) cudaGraphSetConditional((cudaGraphConditionalHandle)P.cond_round, more ? 1u : 0u);
}

__global__ void class_gate_kernel(ClassGateParams P) {
    const int cl = P.first_gated + threadIdx.x;
    if (cl < kQpClasses) cudaGraphSetConditional((cudaGraphConditionalHandle)P.cond[cl], P.order_count[cl] > 0 ? 1u : 0u);
}

cudaError_t launch_class_gate(const ClassGateParams& P, cudaStream_t stream) {
    class_gate_kernel<<<1, 32, 0, stream>>>(P);
    return cudaGetLastError();
}

cudaError_t launch_round_end(const RoundEndParams& P, cudaStream_t stream) {
    round_end_kernel<<<1, 32, 0, stream>>>(P);
    return cudaGetLastError();
}

constexpr int kMinB0 = 6, kMinB1 = 3;    // resident CTAs per SM the small / medium instantiations are compiled for

cudaError_t launch_utility_qp(const QpParams& P, int grid, int cls, cudaStream_t stream) {
    using S0 = QpSmem<32, 128>;
    using S1 = QpSmem<64, 256>;
    using S2 = QpSmem<kWMax, 256>;
    auto k0 = utility_qp_kernel<32, 128, 1, kMinB0>;
    auto k1 = utility_qp_kernel<64, 256, 2, kMinB1>;
    auto k2 = utility_qp_kernel<kWMax, 256, 3, 1>;
    // function attributes are per device: set once for every device this process launches on
    static int n_sm_dev[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    dev &= 63;
    if (!n_sm_dev[dev]) {
        int n = 0;
        e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(S1));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(S2));
        // many small CTAs per SM: ask for the largest shared-memory carve-out
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k0, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k1, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        n_sm_dev[dev] = n;
    }
    if (grid <= 0) return cudaSuccess;
    const int n_sm = n_sm_dev[dev];
    // at most one wave of resident CTAs; they pull columns from the class queue
    if (cls == 1) k0<<<std::min(grid, n_sm * kMinB0), 128, sizeof(S0), stream>>>(P);
    else if (cls == 2) k1<<<std::min(grid, n_sm * kMinB1), 256, sizeof(S1), stream>>>(P);
    else if (cls == 3) k2<<<std::min(grid, n_sm), 256, sizeof(S2), stream>>>(P);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

}  // namespace revs
