// Bracket of the centralized optimum, zone by zone (revs_central_bracket): a voltage-feasible binary schedule (upper
// bound UB_z) and a Lagrangian lower bound LB_z on the cost of every such schedule.
//
// Notation: u = vhigh^2 - vset^2, c the tariff, P = load + rating e with e binary inside the plug-in window and
// n_min <= sum e <= n_max (the SOC window of home_solve), D = R P at the residences, y >= 0 one price per
// (residence, step).  R is block-diagonal over zones, so every zone runs on its own:
//   1. priced selection e*(y): every home takes the n_min window hours of smallest reduced cost
//      rating_h (c_t + (R y)_h,t), then further hours while the reduced cost is negative, up to n_max; ties to the
//      earliest hour, exact values (no grid).  One warp per home (central_select_kernel); R y comes from the network
//      check (network_check_kernel) with y as its schedule.
//   2. Lagrangian value phi(y) = sum c P(y) + sum y (R P(y) - u): a lower bound on the cost of every feasible
//      schedule, at every y.  Per-zone sums in a fixed order (central_ascent_kernel, cen_block_sum).
//   3. start: y = 0, so phi(0) is the cost of every home's cheapest SOC-feasible hours (bench.objective_check's bound
//      of the zone); the greedy repair (repair.cu) of e*(0) gives UB_z, +inf when it leaves violated rows.
//   4. ascent, k = 0 .. iters: evaluate phi(y_k); a larger value than every earlier one is the new best (LB_z, y_best);
//      theta_z (from 1) halves after 20 evaluations without a new best.  The zone stops when UB_z - LB_z <=
//      1e-9 |UB_z|, when the projected subgradient g (G = R P - u; g = G where y > 0, max(G, 0) where y = 0) is 0, when
//      no feasible schedule is known and LB_z > C_max_z, or at k = iters.  Otherwise
//          y <- max(y + alpha_z G, 0),   alpha_z = theta_z (target_z - phi_z) / ||g_z||^2,
//      target_z = UB_z when a feasible schedule is known, else C_max_z + 0.01 |C_max_z|: a value above the cost of
//      every SOC-feasible schedule, so that the bound of a zone without one can pass C_max_z.
//      C_max_z is the cost of the most expensive SOC-feasible schedule: the priced selection of step 1 with reduced
//      cost -rating_h c_t (n_min dearest window hours, then further hours while c_t > 0, up to n_max).
//   5. second start: the repair of e*(y_best); the cheaper of the two repaired schedules is kept, ties to y = 0.
//   6. status: 0 = e*(0) meets every row (optimal, LB = UB); 1 = bracketed; 2 = no feasible schedule found
//      (UB = +inf); 3 = certified infeasible, LB_z > C_max_z: no SOC-feasible schedule meets the rows.
//
// Every value uses explicit round-to-nearest operations and every sum a fixed order (each thread a strided run of the
// zone's [n][T] elements, a warp butterfly, the warps in order), so the result equals the numpy model of
// tests/central_ref.py bit for bit and two calls give the same bytes.
#include <cmath>

#include "kernels.cuh"

namespace revs {

namespace {

constexpr int kCenThreads = 256;
constexpr int kCenWarps = kCenThreads / 32;
constexpr int kCenStall = 20;       // evaluations without a new best before theta halves

// block-wide sum of the threads' partials in a fixed order; valid in thread 0
__device__ __forceinline__ double cen_block_sum(double v, double* slot) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) slot[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = slot[0];
    for (int w = 1; w < kCenWarps; ++w) s = __dadd_rn(s, slot[w]);
    return s;
}

}  // namespace

template <int SLOTS>
__global__ void __launch_bounds__(256, 4) central_select_kernel(CenSelectParams p) {
    const int lane = threadIdx.x & 31;
    const int h = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (h >= p.Hp) return;
    const int T = p.T;
    const size_t base = (size_t)h * T;
    if (!p.has_ev[h]) {                                   // warp-uniform
        for (int t = lane; t < T; t += 32) {
            p.P[base + t] = __dadd_rn(p.load[base + t], 0.0);
            p.p_ev[base + t] = 0.0;
        }
        return;
    }
    const double rate = p.rating[h];
    const int st = p.start[h], en = p.end[h], nmin = p.n_min[h], nmax = p.n_max[h];
    const double* ry = nullptr;                           // (R y) of this residence, step stride n
    int n = 0;
    if (p.ry) {
        const NetZone z = p.zones[p.hzone[h]];
        ry = p.ry + z.home_row * T + (h - z.home_row);
        n = z.n_res;
    }
    double r[SLOTS];
#pragma unroll
    for (int j = 0; j < SLOTS; ++j) {
        const int t = lane + 32 * j;
        double v = INFINITY;
        if (t < T && t >= st && t < en) {
            const double c = p.cost[t];
            v = __dmul_rn(rate, ry ? __dadd_rn(c, ry[(size_t)t * n]) : c);
            if (p.most_expensive) v = -v;
        }
        r[j] = v;
    }
    int in_window = 0;
#pragma unroll
    for (int j = 0; j < SLOTS; ++j) in_window += __popc(__ballot_sync(0xffffffffu, r[j] < INFINITY));
    if ((nmin > nmax || nmin > in_window) && lane == 0) atomicExch(p.infeasible, 1);
    // rank[j] = #{hours s : r_s < r_t or (r_s == r_t and s < t)}
    int rank[SLOTS];
#pragma unroll
    for (int j = 0; j < SLOTS; ++j) rank[j] = 0;
#pragma unroll
    for (int js = 0; js < SLOTS; ++js)
        for (int src = 0; src < 32; ++src) {
            const double o = __shfl_sync(0xffffffffu, r[js], src);
            const int s = src + 32 * js;
#pragma unroll
            for (int j = 0; j < SLOTS; ++j) rank[j] += (o < r[j]) || (o == r[j] && s < lane + 32 * j);
        }
#pragma unroll
    for (int j = 0; j < SLOTS; ++j) {
        const int t = lane + 32 * j;
        if (t >= T) continue;
        const bool on = r[j] < INFINITY && (rank[j] < nmin || (rank[j] < nmax && r[j] < 0.0));
        const double pe = on ? rate : 0.0;
        p.P[base + t] = __dadd_rn(p.load[base + t], pe);
        p.p_ev[base + t] = pe;
    }
}

// One CTA per zone: the Lagrangian value and the projected subgradient norm of the evaluation k, the zone's
// bookkeeping (best bound, theta, stop), then y_best <- y on a new best and y <- max(y + alpha G, 0) on a step.
__global__ void __launch_bounds__(kCenThreads) central_ascent_kernel(CenAscentParams p) {
    __shared__ double slot[3][kCenWarps];
    __shared__ double s_alpha;
    __shared__ int s_best, s_step;
    const int zi = blockIdx.x;
    CenZone* zs = p.state + zi;
    if (p.k > 0 && zs->done) return;
    const NetZone z = p.zones[zi];
    const int n = z.n_res, T = p.T;
    const int64_t m = (int64_t)n * T, row = z.home_row * T;
    const double* __restrict__ Pz = p.P + row;
    const double* __restrict__ Dz = p.D + row;            // [T][n]
    double* yz = p.y + row;
    double a = 0.0, b = 0.0, g2 = 0.0;
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
        const int h = (int)(j / T), t = (int)(j % T);
        const double G = __dadd_rn(Dz[(int64_t)t * n + h], -p.u);
        const double y = yz[j];
        const double g = y > 0.0 ? G : (G > 0.0 ? G : 0.0);
        a = __dadd_rn(a, __dmul_rn(p.cost[t], Pz[j]));
        b = __dadd_rn(b, __dmul_rn(y, G));
        g2 = __dadd_rn(g2, __dmul_rn(g, g));
    }
    a = cen_block_sum(a, slot[0]);
    b = cen_block_sum(b, slot[1]);
    g2 = cen_block_sum(g2, slot[2]);
    if (threadIdx.x == 0) {
        CenZone s = *zs;
        if (p.k == 0) {
            s.lb = -INFINITY;
            s.ub = p.info1[3 * (size_t)zi] == 2 ? INFINITY : p.cost1[zi];
            s.theta = 1.0;
            s.stall = s.done = s.steps = 0;
        }
        const double phi = __dadd_rn(a, b), cm = p.cmax[zi];
        int best = 0;
        if (phi > s.lb) {
            s.lb = phi;
            s.stall = 0;
            best = 1;
        } else if (++s.stall == kCenStall) {
            s.theta *= 0.5;
            s.stall = 0;
        }
        const bool known = s.ub < INFINITY;
        const bool stop = p.k >= p.iters || !(g2 > 0.0) ||
                          (known ? __dadd_rn(s.ub, -s.lb) <= __dmul_rn(1e-9, fabs(s.ub)) : s.lb > cm);
        double alpha = 0.0;
        if (!stop) {
            const double target = known ? s.ub : __dadd_rn(cm, __dmul_rn(0.01, fabs(cm)));
            alpha = __ddiv_rn(__dmul_rn(s.theta, __dadd_rn(target, -phi)), g2);
            ++s.steps;
        }
        s.done = stop;
        *zs = s;
        s_alpha = alpha;
        s_best = best;
        s_step = !stop;
    }
    __syncthreads();
    const int best = s_best, step = s_step;
    const double alpha = s_alpha;
    if (!best && !step) return;
    double* ybz = p.ybest + row;
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
        const double y = yz[j];
        if (best) ybz[j] = y;
        if (step) {
            const int h = (int)(j / T), t = (int)(j % T);
            const double v = __dadd_rn(y, __dmul_rn(alpha, __dadd_rn(Dz[(int64_t)t * n + h], -p.u)));
            yz[j] = v > 0.0 ? v : 0.0;
        }
    }
}

// One CTA per zone: out[z] = sum c P over the zone, in the order of central_ascent_kernel's sum c P.
__global__ void __launch_bounds__(kCenThreads) central_cost_kernel(const NetZone* __restrict__ zones,
                                                                     const double* __restrict__ cost,
                                                                     const double* __restrict__ P, int T,
                                                                     double* __restrict__ out) {
    __shared__ double slot[kCenWarps];
    const NetZone z = zones[blockIdx.x];
    const int64_t m = (int64_t)z.n_res * T;
    const double* __restrict__ Pz = P + z.home_row * T;
    double a = 0.0;
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) a = __dadd_rn(a, __dmul_rn(cost[j % T], Pz[j]));
    a = cen_block_sum(a, slot);
    if (threadIdx.x == 0) out[blockIdx.x] = a;
}

// One CTA per zone: the kept start (the repair of e*(y_best) when strictly cheaper, else the repair of e*(0)), its
// rows copied into P1 / p_ev1, the status, bounds and info.
__global__ void __launch_bounds__(kCenThreads) central_final_kernel(CenFinalParams p) {
    __shared__ int s_take2;
    const int zi = blockIdx.x;
    const NetZone z = p.zones[zi];
    if (threadIdx.x == 0) {
        const int32_t* i1 = p.info1 + 3 * (size_t)zi;
        const int32_t* i2 = p.info2 + 3 * (size_t)zi;
        const double ub1 = i1[0] == 2 ? INFINITY : p.cost1[zi], ub2 = i2[0] == 2 ? INFINITY : p.cost2[zi];
        const int take2 = ub2 < ub1;
        const double ub = take2 ? ub2 : ub1, lb = p.state[zi].lb;
        const int status = i1[0] == 0 ? 0 : ub < INFINITY ? 1 : lb > p.cmax[zi] ? 3 : 2;
        p.bounds[2 * (size_t)zi] = lb;
        p.bounds[2 * (size_t)zi + 1] = ub;
        p.info[3 * (size_t)zi] = status;
        p.info[3 * (size_t)zi + 1] = p.state[zi].steps;
        p.info[3 * (size_t)zi + 2] = take2 ? i2[1] + i2[2] : i1[1] + i1[2];
        s_take2 = take2;
    }
    __syncthreads();
    if (!s_take2) return;
    const int64_t m = (int64_t)z.n_res * p.T, row = z.home_row * p.T;
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
        p.P1[row + j] = p.P2[row + j];
        p.p_ev1[row + j] = p.p_ev2[row + j];
    }
}

cudaError_t launch_central_select(const CenSelectParams& P, cudaStream_t s) {
    if (P.Hp == 0) return cudaSuccess;
    const int warps = 8;
    const dim3 grid((unsigned)((P.Hp + warps - 1) / warps)), block(32 * warps);
    const int slots = (P.T + 31) / 32;
    if (slots <= 1) central_select_kernel<1><<<grid, block, 0, s>>>(P);
    else if (slots <= 3) central_select_kernel<3><<<grid, block, 0, s>>>(P);
    else if (slots <= 8) central_select_kernel<8><<<grid, block, 0, s>>>(P);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

cudaError_t launch_central_ascent(const CenAscentParams& P, int n_zones, cudaStream_t s) {
    if (n_zones == 0) return cudaSuccess;
    central_ascent_kernel<<<n_zones, kCenThreads, 0, s>>>(P);
    return cudaGetLastError();
}

cudaError_t launch_central_cost(const NetZone* zones, int n_zones, const double* cost, const double* P, int T,
                                double* out, cudaStream_t s) {
    if (n_zones == 0) return cudaSuccess;
    central_cost_kernel<<<n_zones, kCenThreads, 0, s>>>(zones, cost, P, T, out);
    return cudaGetLastError();
}

cudaError_t launch_central_final(const CenFinalParams& P, int n_zones, cudaStream_t s) {
    if (n_zones == 0) return cudaSuccess;
    central_final_kernel<<<n_zones, kCenThreads, 0, s>>>(P);
    return cudaGetLastError();
}

}  // namespace revs
