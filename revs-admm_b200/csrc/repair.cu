// Greedy voltage repair of the homes' schedule (revs_repair_schedule): the binary charging decisions of the last ADMM
// run, changed as little as the rule below allows, so that the residences' voltage rows (R P)_i,t <= u hold.
//
// R is block-diagonal over zones: one CTA repairs one zone.  With D = R P at the residences (time-major [T][n] in a
// global scratch, left there by network_check_kernel) and a row (i, t) violated when D[i,t] - u > row_tol:
//   1. take the worst violated row (i*, t*) of the steps not marked stuck (largest excess, then lowest residence,
//      then lowest step -- the order of revs_network_check); stop when there is none;
//   2. candidates: the homes charging at t*, by relief rating_h R[i*,h] descending, ties to the lowest home, with
//      R[i,h] = 2 cumr[lca(node i, node h)] walked on the breadth-first tree of the network check;
//   3. the first candidate with count > n_min drops hour t*; one at count == n_min moves it to the cheapest hour t' of
//      its window it does not charge at and that stays feasible, max_i D[i,t'] + rating_h R[i,h] - u <= row_tol
//      (ties: earliest hour); the first drop or move found is applied (D[:,t*], D[:,t'] and their worst rows are
//      recomputed) and the loop goes back to 1;
//   4. when no candidate can drop or move, t* is marked stuck.
// Charges only leave violated steps and only enter steps that stay feasible, so no feasible step becomes violated and
// every drop or move removes a charge from a violated step: the loop ends.  It is a heuristic -- it does not find the
// cheapest feasible schedule, and a zone may be left with violated rows (status 2; e.g. the base load alone
// violates a row).
//
// Every value is computed with explicit round-to-nearest operations and every maximum under a total order, so the
// result equals the numpy model of tests/repair_ref.py bit for bit.  The zone's small state (per-step worst rows,
// stuck flags, hour bits, relief and R column) lives in shared memory; zones above kRepairSmemMaxN residences (tree-only
// zones) keep it in a global scratch instead.
#include <climits>
#include <cmath>

#include "kernels.cuh"

namespace revs {

namespace {

constexpr int kRepThreads = 256;
constexpr int kRepWarps = kRepThreads / 32;

struct RepArg { double v; int i; };

// larger value first, ties to the lower index
__device__ __forceinline__ bool rep_better(double av, int ai, double bv, int bi) {
    return av > bv || (av == bv && ai < bi);
}

// block-wide arg-max of (v, i); every thread gets the result
__device__ __forceinline__ RepArg rep_argmax(double v, int i, RepArg* slot) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double bv = __shfl_xor_sync(0xffffffffu, v, o);
        const int bi = __shfl_xor_sync(0xffffffffu, i, o);
        if (rep_better(bv, bi, v, i)) { v = bv; i = bi; }
    }
    if ((threadIdx.x & 31) == 0) slot[threadIdx.x >> 5] = RepArg{v, i};
    __syncthreads();
    if (threadIdx.x == 0) {
        RepArg m = slot[0];
        for (int w = 1; w < kRepWarps; ++w)
            if (rep_better(slot[w].v, slot[w].i, m.v, m.i)) m = slot[w];
        slot[kRepWarps] = m;
    }
    __syncthreads();
    const RepArg r = slot[kRepWarps];
    __syncthreads();
    return r;
}

// The zone's state, in shared memory or in the global scratch (layout of repair_ws_bytes).
struct RepWs {
    double *wv, *rel, *col;   // [T] worst excess of every step, [n] relief of the candidates, [n] R column * rating
    uint64_t* bits;           // [n][W] hour bits
    int *wi, *ord, *stuck;    // [T] residence of the worst excess, steps by (cost, step), stuck flags
    int* hpos;                // [n] breadth-first position of every residence's node
};

__host__ __device__ inline size_t rep_take(size_t& o, size_t bytes) {
    const size_t at = o;
    o += (bytes + 15) & ~(size_t)15;
    return at;
}

__host__ __device__ inline size_t rep_layout(int n, int T, char* base, RepWs* w) {
    const int W = (T + 63) / 64;
    size_t o = 0;
    const size_t wv = rep_take(o, sizeof(double) * T), rel = rep_take(o, sizeof(double) * n),
                 col = rep_take(o, sizeof(double) * n), bits = rep_take(o, sizeof(uint64_t) * n * W),
                 wi = rep_take(o, sizeof(int) * T), ord = rep_take(o, sizeof(int) * T), stuck = rep_take(o, sizeof(int) * T),
                 hpos = rep_take(o, sizeof(int) * n);
    if (w) {
        w->wv = (double*)(base + wv); w->rel = (double*)(base + rel); w->col = (double*)(base + col);
        w->bits = (uint64_t*)(base + bits); w->wi = (int*)(base + wi); w->ord = (int*)(base + ord);
        w->stuck = (int*)(base + stuck); w->hpos = (int*)(base + hpos);
    }
    return o;
}

// worst excess of step t (largest D - u, lowest residence)
__device__ __forceinline__ void rep_step_worst(const double* __restrict__ Dt, int n, double u, int t, const RepWs& w, RepArg* slot) {
    double v = -INFINITY;
    int i = INT_MAX;
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
        const double x = __dadd_rn(Dt[k], -u);
        if (rep_better(x, k, v, i)) { v = x; i = k; }
    }
    const RepArg m = rep_argmax(v, i, slot);
    if (threadIdx.x == 0) { w.wv[t] = m.v; w.wi[t] = m.i; }
}

}  // namespace

__global__ void __launch_bounds__(kRepThreads, 2) repair_kernel(RepairParams p) {
    extern __shared__ __align__(16) char rep_smem[];
    __shared__ RepArg slot[kRepWarps + 1];
    __shared__ int s_t, s_i;
    const int zi = blockIdx.x;
    const NetZone z = p.zones[zi];
    const int n = z.n_res, T = p.T, W = (T + 63) / 64;
    int32_t* info = p.info + 3 * (size_t)zi;
    if (!(p.zone_worst[3 * (size_t)zi + 1] > p.row_tol)) {        // no violated row: the zone is untouched
        if (threadIdx.x == 0) { info[0] = 0; info[1] = 0; info[2] = 0; }
        return;
    }
    RepWs w;
    rep_layout(n, T, p.ws_off[zi] < 0 ? rep_smem : p.gws + p.ws_off[zi], &w);
    const NetNode* __restrict__ nd = p.nodes + z.node0;
    const int* __restrict__ rl = p.res + z.res0;
    const double* __restrict__ cumr = p.cumr + z.out_row;
    double* D = p.D + z.home_row * T;                             // [T][n]
    const int64_t h0 = z.home_row;
    const double u = p.u, tol = p.row_tol;

    for (int q = threadIdx.x; q < z.n_nodes; q += blockDim.x) {
        const NetNode a = nd[q];
        for (int e = 0; e < a.nres; ++e) w.hpos[rl[a.res0 + e]] = q;
    }
    for (int k = threadIdx.x; k < n * W; k += blockDim.x) {
        const int h = k / W, t0 = 64 * (k % W);
        const double* pe = p.p_ev + (h0 + h) * T;
        uint64_t b = 0;
        for (int t = t0; t < min(T, t0 + 64); ++t)
            if (pe[t] > 0.0) b |= 1ull << (t - t0);
        w.bits[k] = b;
    }
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        const double c = p.cost[t];
        int r = 0;
        for (int s = 0; s < T; ++s) r += p.cost[s] < c || (p.cost[s] == c && s < t);
        w.ord[r] = t;
        w.stuck[t] = 0;
    }
    __syncthreads();
    for (int t = 0; t < T; ++t) rep_step_worst(D + (size_t)t * n, n, u, t, w, slot);
    __syncthreads();

    int moves = 0, drops = 0;                                     // thread 0
    for (;;) {
        // 1. worst violated row of the steps not stuck
        if (threadIdx.x < 32) {
            double v = -INFINITY;
            int i = INT_MAX, ts = INT_MAX;
            for (int t = threadIdx.x; t < T; t += 32) {
                if (w.stuck[t] || !(w.wv[t] > tol)) continue;
                const double x = w.wv[t];
                const int r = w.wi[t];
                if (x > v || (x == v && (r < i || (r == i && t < ts)))) { v = x; i = r; ts = t; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double bv = __shfl_xor_sync(0xffffffffu, v, o);
                const int bi = __shfl_xor_sync(0xffffffffu, i, o), bt = __shfl_xor_sync(0xffffffffu, ts, o);
                if (bv > v || (bv == v && (bi < i || (bi == i && bt < ts)))) { v = bv; i = bi; ts = bt; }
            }
            if (threadIdx.x == 0) { s_t = ts == INT_MAX ? -1 : ts; s_i = i; }
        }
        __syncthreads();
        const int ts = s_t, is = s_i;
        if (ts < 0) break;
        // 2. relief of the homes charging at ts
        const int qi = w.hpos[is];
        for (int h = threadIdx.x; h < n; h += blockDim.x)
            w.rel[h] = (w.bits[h * W + (ts >> 6)] >> (ts & 63)) & 1ull
                           ? __dmul_rn(p.rating[h0 + h], lca_r(nd, cumr, qi, w.hpos[h])) : -INFINITY;
        __syncthreads();
        // 3. candidates in order of relief: the first that can drop or move
        int act = 0, tp = -1, hc = -1;
        for (;;) {
            double cv = -INFINITY;
            int ci = INT_MAX;
            for (int h = threadIdx.x; h < n; h += blockDim.x)
                if (rep_better(w.rel[h], h, cv, ci)) { cv = w.rel[h]; ci = h; }
            const RepArg c = rep_argmax(cv, ci, slot);
            if (c.v == -INFINITY) break;
            hc = c.i;
            const double rt = p.rating[h0 + hc];
            const int qh = w.hpos[hc];
            for (int i = threadIdx.x; i < n; i += blockDim.x) w.col[i] = __dmul_rn(rt, lca_r(nd, cumr, w.hpos[i], qh));
            int cnt = 0;
            for (int k = 0; k < W; ++k) cnt += __popcll(w.bits[hc * W + k]);
            if (cnt > p.n_min[h0 + hc]) {
                act = 1;
            } else {
                const int st = p.start[h0 + hc], en = p.end[h0 + hc];
                for (int k = 0; k < T; ++k) {
                    const int t = w.ord[k];
                    if (t < st || t >= en || ((w.bits[hc * W + (t >> 6)] >> (t & 63)) & 1ull)) continue;
                    const double* Dt = D + (size_t)t * n;
                    int bad = 0;
                    for (int i = threadIdx.x; i < n; i += blockDim.x)
                        bad |= __dadd_rn(__dadd_rn(Dt[i], w.col[i]), -u) > tol;
                    if (!__syncthreads_or(bad)) { tp = t; act = 2; break; }
                }
            }
            __syncthreads();
            if (act) break;
            if (threadIdx.x == 0) w.rel[hc] = -INFINITY;          // tried
            __syncthreads();
        }
        if (!act) {                                               // 4. nothing can leave ts
            if (threadIdx.x == 0) w.stuck[ts] = 1;
            __syncthreads();
            continue;
        }
        double* Ds = D + (size_t)ts * n;
        double* Dp = tp >= 0 ? D + (size_t)tp * n : nullptr;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            Ds[i] = __dadd_rn(Ds[i], -w.col[i]);
            if (Dp) Dp[i] = __dadd_rn(Dp[i], w.col[i]);
        }
        if (threadIdx.x == 0) {
            const int64_t row = (h0 + hc) * T;
            w.bits[hc * W + (ts >> 6)] &= ~(1ull << (ts & 63));
            p.P[row + ts] = __dadd_rn(p.load[row + ts], 0.0);
            p.p_ev[row + ts] = 0.0;
            if (tp >= 0) {
                const double rt = p.rating[h0 + hc];
                w.bits[hc * W + (tp >> 6)] |= 1ull << (tp & 63);
                p.P[row + tp] = __dadd_rn(p.load[row + tp], rt);
                p.p_ev[row + tp] = rt;
                ++moves;
            } else {
                ++drops;
            }
        }
        __syncthreads();
        rep_step_worst(Ds, n, u, ts, w, slot);
        if (Dp) rep_step_worst(Dp, n, u, tp, w, slot);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int left = 0;
        for (int t = 0; t < T; ++t) left |= w.stuck[t];
        info[0] = left ? 2 : 1;
        info[1] = moves;
        info[2] = drops;
    }
}

size_t repair_ws_bytes(int n, int T) { return rep_layout(n, T, nullptr, nullptr); }

cudaError_t launch_repair(const RepairParams& P, int n_zones, size_t smem, cudaStream_t s) {
    if (n_zones == 0) return cudaSuccess;
    // always the same value: solvers of one device may launch from several host threads at once
    cudaError_t e = cudaFuncSetAttribute(repair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)repair_ws_bytes(kRepairSmemMaxN, kRepairMaxT));
    if (e != cudaSuccess) return e;
    repair_kernel<<<n_zones, kRepThreads, smem, s>>>(P);
    return cudaGetLastError();
}

}  // namespace revs
