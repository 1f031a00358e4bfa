// Certificate of voltage infeasibility, zone by zone (revs_certify_infeasible): a proof that no binary schedule keeps
// every home's SOC window and plug-in window and the residences' voltage rows (R P)_i,t - u <= row_tol.
//
// The Lagrangian bound of revs_central_bracket cannot give this proof whenever the LP relaxation meets the rows: every
// home's set {e in [0,1], n_min <= sum e <= n_max, inside the window} is an integral polytope, so the dual equals the
// LP bound.  The binary program can still be infeasible, because a home draws its full rating in every hour it charges.
// The rule counts charges.  Notation: D0 = R load at the residences (network_check_kernel, its order),
// a_h(i) = rating_h R[i,h] (lca_r), the homes that count are the EV homes with n_min > 0, thr = row_tol + 1e-12, and a
// set of charges fits row (i,t) when (D0[i,t] + s) - u <= thr, s the sum of their coefficients added in ascending
// order.  The 1e-12 pu^2 margin resolves every rounding in favour of "fits", so no certificate comes from rounding.
//   kind 1: some row has D0[i,t] - u > thr (the base load alone violates it); the witness is the worst row (largest
//           excess, then lowest residence, then lowest step).
//   kind 2: for a residence i, S_k = the k homes of largest a_h(i) (ties to the lowest home), k = 1..K,
//           K = min(kCertTopK, homes that count).  At step t at most m_t(k) members of S_k charge, m_t(k) the largest j
//           such that the j smallest coefficients of the members whose window contains t fit row (i,t): any j members
//           charging at t have a sum at least as large, and R >= 0, rating >= 0 mean that other charges only use up
//           slack.  So cap_k = sum_t m_t(k) < need_k = sum_{S_k} n_min proves the zone infeasible.  The witness is the
//           (i, k) of the largest need_k - cap_k, then lowest residence, then lowest k.
//
// Three launches: certify_base_kernel (one CTA per zone: kind 1, breadth-first positions of the residences, window and
// rating checks), certify_count_kernel (one warp per residence row: the top-K coefficients in registers, the step loop
// over shared memory; the rows of a zone meet in a 64-bit atomicMax of the packed witness) and certify_final_kernel.
// Every value uses explicit round-to-nearest operations and every reduction is an integer or total-order maximum, so
// the result is exact, deterministic and equal to the numpy model of tests/certify_ref.py.  No state is kept per zone
// beyond one [Hp] array of positions, so zones of any size (tree-only zones) run the same code.
#include <climits>
#include <cmath>

#include "kernels.cuh"

namespace revs {

namespace {

constexpr int kCertThreads = 256;
constexpr int kCertWarps = kCertThreads / 32;
static_assert(kCertTopK == 32, "the top-K list holds one home per lane");

// larger value first, ties to the lower index
__device__ __forceinline__ bool cert_better(double av, long long ai, double bv, long long bi) {
    return av > bv || (av == bv && ai < bi);
}

// witness of kind 2 as one 64-bit word whose unsigned maximum is the witness order: need - cap (< 2^24: n_min <= T <=
// kRepairMaxT, K <= 32), then the lowest residence, then the lowest k
__device__ __forceinline__ unsigned long long cert_key(int deficit, int i, int k) {
    return ((unsigned long long)deficit << 40) | ((unsigned long long)(0xffffffffu - (unsigned)i) << 8) |
           (unsigned long long)(255 - k);
}

}  // namespace

// One CTA per zone: the zone's worst base-load row (kind 1), the breadth-first position of every residence's node
// (for certify_count_kernel), the checks of its homes and the reset of its witness word.
__global__ void __launch_bounds__(kCertThreads) certify_base_kernel(CertParams p) {
    __shared__ double sv[kCertWarps];
    __shared__ long long sl[kCertWarps];
    const int zi = blockIdx.x;
    const NetZone z = p.zones[zi];
    const int n = z.n_res, T = p.T;
    const int64_t h0 = z.home_row;
    const NetNode* __restrict__ nd = p.nodes + z.node0;
    const int* __restrict__ rl = p.res + z.res0;
    for (int q = threadIdx.x; q < z.n_nodes; q += blockDim.x) {
        const NetNode a = nd[q];
        for (int e = 0; e < a.nres; ++e) p.hpos[h0 + rl[a.res0 + e]] = q;
    }
    for (int h = threadIdx.x; h < n; h += blockDim.x) {
        if (!p.has_ev[h0 + h]) continue;
        const double r = p.rating[h0 + h];
        if (!(r >= 0.0 && r < INFINITY)) atomicOr(p.flag, 2);
        const int st = max(p.start[h0 + h], 0), en = min(p.end[h0 + h], T), nmin = p.n_min[h0 + h];
        if (nmin > p.n_max[h0 + h] || nmin > max(en - st, 0)) atomicOr(p.flag, 1);
    }
    // worst row of the base load: largest D0 - u, then lowest loc = i T + t
    const double* __restrict__ D = p.D + h0 * T;                  // [T][n]
    double v = -INFINITY;
    long long l = LLONG_MAX;
    for (int64_t j = threadIdx.x; j < (int64_t)n * T; j += blockDim.x) {
        const int t = (int)(j / n), i = (int)(j % n);
        const double x = __dadd_rn(D[j], -p.u);
        const long long lj = (long long)i * T + t;
        if (cert_better(x, lj, v, l)) { v = x; l = lj; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double bv = __shfl_xor_sync(0xffffffffu, v, o);
        const long long bl = __shfl_xor_sync(0xffffffffu, l, o);
        if (cert_better(bv, bl, v, l)) { v = bv; l = bl; }
    }
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = v; sl[threadIdx.x >> 5] = l; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kCertWarps; ++w)
            if (cert_better(sv[w], sl[w], v, l)) { v = sv[w]; l = sl[w]; }
        int32_t* c = p.cert + 4 * (size_t)zi;
        const bool base = v > p.thr;
        c[0] = base ? 1 : 0;
        c[1] = base ? (int32_t)(l / T) : -1;
        c[2] = base ? (int32_t)(l % T) : -1;
        c[3] = 0;
        p.key[zi] = 0;
    }
}

// One warp per residence row (padded home rows; padding and zones of kind 1 exit at once).
__global__ void __launch_bounds__(kCertThreads) certify_count_kernel(CertParams p) {
    __shared__ double sd[kCertWarps][kRepairMaxT];                 // D0[i, t] of the warp's row
    __shared__ double sa[kCertWarps][kCertTopK];                   // the row's top-K coefficients, descending
    __shared__ int sst[kCertWarps][kCertTopK], sen[kCertWarps][kCertTopK];
    const int wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kCertWarps + wp;
    if (row >= p.Hp) return;                                      // warp-uniform from here on
    const int zi = p.hzone[row];
    if (zi < 0 || p.cert[4 * (size_t)zi] == 1) return;
    const NetZone z = p.zones[zi];
    const int n = z.n_res, T = p.T;
    const int64_t h0 = z.home_row;
    const int i = (int)(row - h0);
    const NetNode* __restrict__ nd = p.nodes + z.node0;
    const double* __restrict__ cumr = p.cumr + z.out_row;
    const int qi = p.hpos[row];

    // top-K of a_h(i) over the homes that count: lane j holds the j-th (value descending, home ascending); a candidate
    // better than the last entry is inserted at its rank and the entries behind it move down one lane
    double v = -INFINITY;
    int hk = INT_MAX;
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int h = c0 + lane;
        double cv = -INFINITY;
        if (h < n && p.has_ev[h0 + h] && p.n_min[h0 + h] > 0)
            cv = __dmul_rn(p.rating[h0 + h], lca_r(nd, cumr, qi, p.hpos[h0 + h]));
        const double lv = __shfl_sync(0xffffffffu, v, 31);
        const int lh = __shfl_sync(0xffffffffu, hk, 31);
        unsigned m = __ballot_sync(0xffffffffu, cv > -INFINITY && cert_better(cv, h, lv, lh));
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            const double x = __shfl_sync(0xffffffffu, cv, b);
            const int xh = c0 + b;
            const unsigned worse = __ballot_sync(0xffffffffu, !cert_better(v, hk, x, xh));
            const double pv = __shfl_up_sync(0xffffffffu, v, 1);
            const int ph = __shfl_up_sync(0xffffffffu, hk, 1);
            if (!worse) continue;
            const int pos = __ffs(worse) - 1;
            if (lane > pos) { v = pv; hk = ph; }
            else if (lane == pos) { v = x; hk = xh; }
        }
    }
    const int K = __popc(__ballot_sync(0xffffffffu, hk != INT_MAX));
    if (K == 0) return;
    int need = 0;
    if (lane < K) {
        sa[wp][lane] = v;
        sst[wp][lane] = p.start[h0 + hk];
        sen[wp][lane] = p.end[h0 + hk];
        need = p.n_min[h0 + hk];
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {                            // need_k = sum of n_min over lanes 0..k-1
        const int x = __shfl_up_sync(0xffffffffu, need, o);
        if (lane >= o) need += x;
    }
    for (int t = lane; t < T; t += 32) sd[wp][t] = p.D[h0 * T + (int64_t)t * n + i];
    __syncwarp();

    // lane k - 1: cap_k; S_k ascending is the ranking backwards from entry k - 1
    unsigned long long key = 0;
    if (lane < K) {
        const int k = lane + 1;
        int cap = 0;
        for (int t = 0; t < T; ++t) {
            const double d = sd[wp][t];
            double s = 0.0;
            for (int r = k - 1; r >= 0; --r) {
                if (t < sst[wp][r] || t >= sen[wp][r]) continue;
                s = __dadd_rn(s, sa[wp][r]);
                if (!(__dadd_rn(__dadd_rn(d, s), -p.u) <= p.thr)) break;
                ++cap;
            }
        }
        if (need > cap) key = cert_key(need - cap, i, k);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long x = __shfl_xor_sync(0xffffffffu, key, o);
        key = x > key ? x : key;
    }
    if (lane == 0 && key) atomicMax(p.key + zi, key);
}

// One thread per zone: the witness of kind 2 from its word, for the zones without a kind 1 certificate.
__global__ void certify_final_kernel(int32_t* __restrict__ cert, const unsigned long long* __restrict__ key, int n_zones) {
    const int zi = blockIdx.x * blockDim.x + threadIdx.x;
    if (zi >= n_zones) return;
    const unsigned long long w = key[zi];
    int32_t* c = cert + 4 * (size_t)zi;
    if (c[0] == 1 || w == 0) return;
    c[0] = 2;
    c[1] = (int32_t)(0xffffffffu - (unsigned)(w >> 8));
    c[2] = 255 - (int)(w & 255);
    c[3] = (int32_t)(w >> 40);
}

cudaError_t launch_certify(const CertParams& P, int n_zones, cudaStream_t s) {
    if (n_zones == 0) return cudaSuccess;
    certify_base_kernel<<<n_zones, kCertThreads, 0, s>>>(P);
    certify_count_kernel<<<(unsigned)((P.Hp + kCertWarps - 1) / kCertWarps), kCertThreads, 0, s>>>(P);
    certify_final_kernel<<<(n_zones + 127) / 128, 128, 0, s>>>(P.cert, P.key, n_zones);
    return cudaGetLastError();
}

}  // namespace revs
