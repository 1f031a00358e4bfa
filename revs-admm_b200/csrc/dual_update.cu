// Fused dual-price update, per-home convergence value, primal/dual residuals, the
// convergence test and the target of the next utility step -- one kernel per ADMM
// iteration, nothing leaves the device.
//
// Reference: the tail of the home loop of solve_ADMM (lpsolver.py:280-284)
//     check = P_est[k+1] - P_sch[k+1]
//     G[k+1] = G[k] + kappa/2 * check
//     diff[k+1][h] = ||check|| / T
// plus the objective data of the next Utility (lpsolver.py:202-204), which is the
// projection target  z = (P_est + P_sch)/2 - G/kappa.
//
// Layout: the utility side keeps its arrays time-major [T][Hp] (one contiguous column per
// (feeder,hour) QP), the home side home-major [Hp][T] (one contiguous row per home).  A
// CTA owns 32 homes x T hours and transposes through shared memory, so both sides are
// read and written in full 256-byte runs.  Per-home norms use warp shuffles; every CTA leaves
// its two partial sums in global memory and the last CTA to finish adds them in a fixed order
// (reproducible residuals), exchanges them with the other GPUs of the box over peer memory
// when peers are attached, and sets the converged flag / the condition of the captured loop.
//
// HBM traffic: 58 bytes per home-step (reads P_est time-major, P_sch[k+1], Gamma; writes Gamma,
// P_est home-major, z, g = [z]_+ and its bf16 copy).  The previous schedule P_sch[k] of the dual
// residual is not read: home_solve_kernel, which had both schedules in registers, leaves the
// per-home sums behind (DualParams::dsum).  The home-major loads of the two homes a warp handles
// together are all issued before the first use (SLOTS = hours per lane at compile time); left to
// the compiler they were three dependent round trips per home (profiles/README_r02.md).
#include <cuda_bf16.h>

#include "kernels.cuh"

namespace revs {



__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// SLOTS = ceil(T / 32) hours per lane, compile-time: every load of a home (and of the second home a warp handles at
// the same time) is issued before the first value is used -- two round trips to HBM per warp instead of twelve.
// SLOTS = 0: any T, run-time loop over the hours.
template <int SLOTS, bool DSUM>
__global__ void __launch_bounds__(256, 4) dual_update_kernel(DualParams P) {
    extern __shared__ double tile[];   // [32][T+1]
    __shared__ double s_part[2][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int h0 = blockIdx.x * 32;
    const int ldt = P.T + 1;
    const int it = P.iter ? *P.iter : 0;          // read by every CTA before the last one increments it (ticket below)
    const double* __restrict__ p_sch_new = (it & 1) ? P.p_sch_old : P.p_sch_new;
    const double* __restrict__ p_sch_old = (it & 1) ? P.p_sch_new : P.p_sch_old;
    double* __restrict__ diff_k = P.diff_k + (size_t)it * P.Hp;

    {
        const int h = h0 + lane;
        const bool in = h < P.Hp;
        const double* src = P.g_t + (in ? h : 0);
        int t = warp;
        for (; t + 24 < P.T; t += 32) {               // four rows of the tile per step: the loads overlap
            double v[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = in ? src[(size_t)(t + 8 * q) * P.Hp] : 0.0;
#pragma unroll
            for (int q = 0; q < 4; ++q) tile[lane * ldt + t + 8 * q] = v[q];
        }
        for (; t < P.T; t += 8) tile[lane * ldt + t] = in ? src[(size_t)t * P.Hp] : 0.0;
    }
    __syncthreads();

    const double hk = 0.5 * P.kappa;
    double blk_p = 0.0, blk_d = 0.0;
    // the sum of (P_sch[k+1] - P_sch[k])^2 of a home comes from home_solve_kernel when it left it behind (dsum): same
    // additions in the same order as the loop below, without reading the previous schedule again
    const double* dsum = DSUM ? P.dsum : nullptr;
    if constexpr (SLOTS > 0) {
        for (int hl = warp; hl < 32; hl += 16) {      // homes hl and hl + 8 of the tile together
            double sn[2][SLOTS], gm[2][SLOTS], so[2][DSUM ? 1 : SLOTS];
            bool okh[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int h = h0 + hl + 8 * q;
                okh[q] = h < P.Hp;
                const size_t base = (size_t)(okh[q] ? h : 0) * P.T;
#pragma unroll
                for (int j = 0; j < SLOTS; ++j) {
                    const int t = min(lane + 32 * j, P.T - 1);
                    sn[q][j] = p_sch_new[base + t];
                    gm[q][j] = P.gamma[base + t];
                    if constexpr (!DSUM) so[q][j] = p_sch_old[base + t];
                }
            }
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                if (!okh[q]) continue;                // warp-uniform
                const int h = h0 + hl + 8 * q;
                const size_t base = (size_t)h * P.T;
                double a1 = 0.0, a2 = 0.0;
#pragma unroll
                for (int j = 0; j < SLOTS; ++j) {
                    const int t = lane + 32 * j;
                    if (t < P.T) {
                        const double e = tile[(hl + 8 * q) * ldt + t];
                        const double check = __dadd_rn(e, -sn[q][j]);
                        const double g2 = __dadd_rn(gm[q][j], __dmul_rn(hk, check));
                        P.gamma[base + t] = g2;
                        P.p_est[base + t] = e;
                        tile[(hl + 8 * q) * ldt + t] = __dadd_rn(__dmul_rn(__dadd_rn(e, sn[q][j]), 0.5), -__ddiv_rn(g2, P.kappa));
                        a1 = fma(check, check, a1);
                        if constexpr (!DSUM) {
                            const double ds = sn[q][j] - so[q][j];
                            a2 = fma(ds, ds, a2);
                        }
                    }
                }
                a1 = warp_sum(a1);
                a2 = DSUM ? dsum[h] : warp_sum(a2);
                if (lane == 0) diff_k[h] = sqrt(a1) / (double)P.T;
                blk_p += a1;
                blk_d += a2;
            }
        }
    } else {
        for (int hl = warp; hl < 32; hl += 8) {
            const int h = h0 + hl;
            if (h >= P.Hp) break;
            const size_t base = (size_t)h * P.T;
            double a1 = 0.0, a2 = 0.0;
            for (int t = lane; t < P.T; t += 32) {
                const double e = tile[hl * ldt + t];
                const double sn = p_sch_new[base + t];
                const double so = dsum ? 0.0 : p_sch_old[base + t];
                const double gm = P.gamma[base + t];
                const double check = __dadd_rn(e, -sn);
                const double g2 = __dadd_rn(gm, __dmul_rn(hk, check));
                P.gamma[base + t] = g2;
                P.p_est[base + t] = e;
                tile[hl * ldt + t] = __dadd_rn(__dmul_rn(__dadd_rn(e, sn), 0.5), -__ddiv_rn(g2, P.kappa));
                a1 = fma(check, check, a1);
                const double ds = sn - so;
                a2 = fma(ds, ds, a2);
            }
            a1 = warp_sum(a1);
            a2 = dsum ? dsum[h] : warp_sum(a2);
            if (lane == 0) diff_k[h] = sqrt(a1) / (double)P.T;
            blk_p += a1;
            blk_d += a2;
        }
    }
    if (lane == 0) { s_part[0][warp] = blk_p; s_part[1][warp] = blk_d; }
    __syncthreads();

    __nv_bfloat16* gbf = reinterpret_cast<__nv_bfloat16*>(P.gbf_next);
    for (int t = warp; t < P.T; t += 8) {
        int h = h0 + lane;
        if (h < P.Hp) {
            const double zv = tile[lane * ldt + t];
            const size_t o = (size_t)t * P.Hp + h;
            P.z_t[o] = zv;
            if (P.g_next) {                    // start of the next utility solve: g = [z]_+ wherever no multiplier is stored
                const double gv = fmax(zv, 0.0);
                P.g_next[o] = gv;
                if (gbf) gbf[o] = __float2bfloat16_rn((float)gv);
            }
        }
    }

    // residuals: per-CTA partial sums, added by the last CTA in a fixed order (no floating-point atomics: the
    // residuals and the convergence decision are reproducible run to run)
    __shared__ int s_last;
    __shared__ double s_fin[2][8];
    if (threadIdx.x == 0) {
        double sp = 0.0, sd = 0.0;
        for (int w = 0; w < 8; ++w) { sp += s_part[0][w]; sd += s_part[1][w]; }
        P.partials[blockIdx.x] = sp;
        P.partials[gridDim.x + blockIdx.x] = sd;
        __threadfence();
        const unsigned done = atomicAdd(&P.res->ticket, 1u);
        s_last = done == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    double tp = 0.0, td = 0.0;
    for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x) {
        tp += __ldcg(P.partials + b);
        td += __ldcg(P.partials + gridDim.x + b);
    }
    tp = warp_sum(tp);
    td = warp_sum(td);
    if (lane == 0) { s_fin[0][warp] = tp; s_fin[1][warp] = td; }
    __syncthreads();
    __shared__ double s_peer[3][kMaxPeers];
    if (P.peer.world > 1) {
        // ---- all-reduce over the GPUs of the box (see PeerReduce): thread r talks to rank r
        const int r = threadIdx.x;
        if (r < P.peer.world) {
            double lp = 0.0, ld = 0.0;
            for (int w = 0; w < 8; ++w) { lp += s_fin[0][w]; ld += s_fin[1][w]; }
            const int pit = P.iter ? it : P.step;       // host-driven loop: the iteration number comes with the launch
            const unsigned long long seq = *P.peer.run_seq + (unsigned long long)pit + 1ull;
            const int par = pit & 1;
            PeerSlot* out = P.peer.box[r] + par * P.peer.world + P.peer.rank;       // my slot in rank r's mailbox
            out->v[0] = lp;
            out->v[1] = ld;
            out->v[2] = P.count;
            __threadfence_system();
            st_release_sys(&out->seq, seq);
            PeerSlot* in = P.peer.box[P.peer.rank] + par * P.peer.world + r;         // rank r's slot in my mailbox
            const long long t0 = clock64();
            bool ok = true;
            while (ld_acquire_sys(&in->seq) != seq) {
                if (clock64() - t0 > 20000000000ll) { ok = false; break; }           // ~10 s: a peer died
                __nanosleep(200);
            }
            if (!ok) atomicExch(P.peer.timeout, 1);
            s_peer[0][r] = ok ? in->v[0] : 0.0;
            s_peer[1][r] = ok ? in->v[1] : 0.0;
            s_peer[2][r] = ok ? in->v[2] : 0.0;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        tp = 0.0; td = 0.0;
        double count = P.count;
        if (P.peer.world > 1) {
            count = 0.0;
            for (int r = 0; r < P.peer.world; ++r) { tp += s_peer[0][r]; td += s_peer[1][r]; count += s_peer[2][r]; }
        } else {
            for (int w = 0; w < 8; ++w) { tp += s_fin[0][w]; td += s_fin[1][w]; }
        }
        const double r = sqrt(tp / count), sres = P.kappa * sqrt(td / count);
        const int conv = (P.tol > 0.0 && r < P.tol && sres < P.tol) ? 1 : 0;
        P.res->sum_primal = tp;                    // global sums when peers are attached
        P.res->sum_dual = td;
        P.res->count = count;
        P.res->primal = r;
        P.res->dual = sres;
        P.res->converged = conv;
        P.res->ticket = 0u;                        // ready for the next iteration of a captured loop
        if (P.iter) {
            const int k = it + 1;
            *P.iter = k;
            if (P.use_cond) {
                const bool err = (P.err_a && *P.err_a) || (P.err_b && *P.err_b) || (P.peer.world > 1 && *P.peer.timeout);
                cudaGraphSetConditional((cudaGraphConditionalHandle)P.cond_loop, (k < P.iter_max && !conv && !err) ? 1u : 0u);
            }
        }
    }
}

cudaError_t launch_dual_update(const DualParams& P, cudaStream_t stream) {
    const size_t smem = (size_t)32 * (P.T + 1) * sizeof(double);
    const int slots = (P.T + 31) / 32;
    const dim3 grid((P.Hp + 31) / 32);
    auto go = [&](auto kernel) -> cudaError_t {
        // the 48 KB a launch gets without opting in hold the kernel's static shared memory too (s_part, s_fin, s_peer:
        // 1.7 KB), so the tile needs the opt-in from T = 185 on, not only beyond 48 KB of its own (T >= 192)
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
        if (e != cudaSuccess) return e;
        if (smem + fa.sharedSizeBytes > 48 * 1024) {
            e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kernel<<<grid, 256, smem, stream>>>(P);
        return cudaGetLastError();
    };
    if (P.dsum) {
        switch (slots) {
            case 1: return go(dual_update_kernel<1, true>);
            case 2: return go(dual_update_kernel<2, true>);
            case 3: return go(dual_update_kernel<3, true>);
            case 4: return go(dual_update_kernel<4, true>);
            default: return go(dual_update_kernel<0, true>);
        }
    }
    switch (slots) {
        case 1: return go(dual_update_kernel<1, false>);
        case 2: return go(dual_update_kernel<2, false>);
        case 3: return go(dual_update_kernel<3, false>);
        case 4: return go(dual_update_kernel<4, false>);
        default: return go(dual_update_kernel<0, false>);
    }
}

}  // namespace revs
