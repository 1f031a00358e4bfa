// Hosting capacity of a schedule (revs_hosting_capacity): for every residence and step, the extra load its home can
// draw, with everything else unchanged, before a voltage row or a line rating binds; for every zone and step, the
// extra load every residence of the zone can draw at once.  Definitions and the exactness argument are in
// include/revs_admm.h.
//
// Per zone and step, on the network check's breadth-first arrays (network_check.cu), four level passes:
//     F_i = inj_i + sum_{children c} F_c                           leaves -> root   (as the network check)
//     D_i = D_parent(i) + 2 r_i F_i                                root -> leaves   (as the network check)
//     M_i = min(sigma_i if residences hang on i, min_c M_c)        leaves -> root   (sigma = (u + row_tol) - D)
//     V_i = min(V_parent(i), M_i / d_i if d_i > 0),  L_i = min(L_parent(i), th_i)   root -> leaves
// with d_i = 2 cumr[i] and th_i = (1 - |s_i| F_i) / |s_i| on rated edges (+inf elsewhere).  A home's capacity is
// max(0, min(V, L)) at its node.  The state of a step is two doubles per node (F, D, M, V in place, and th, then L in
// place): the hosting CTAs have their own step grouping, and a zone whose one-step state does not fit in shared
// memory runs on a global scratch, as in the network check.
//
// Every thread of a CTA works on one step (the block size is a multiple of the steps per CTA), so the zone's uniform
// headroom of a step is a minimum over the threads of that step, and one CTA owns each (zone, step).  Minima and
// integer counts do not depend on the order of their operands: the outputs are the same for any CTA schedule, and the
// per-value arithmetic is that of the numpy model of tests/hosting_ref.py, bit for bit.
#include <algorithm>
#include <cmath>

#include "kernels.cuh"

namespace revs {

namespace {

constexpr int kHcThreads = 256;
constexpr int kHcWarps = kHcThreads / 32;
// the final per-step minima and counts of the warps, in the dynamic shared memory once the state is no longer read (a
// static array would keep two CTAs of 112 KB of state from sharing an SM)
constexpr size_t kHcScratch = kHcWarps * (32 * sizeof(double) + 3 * sizeof(unsigned long long));

__device__ __forceinline__ unsigned long long hc_sum(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace

__global__ void __launch_bounds__(kHcThreads) hosting_kernel(HcParams p, const int* __restrict__ list) {
    extern __shared__ double hc_smem[];
    const int cid = list[blockIdx.x];
    const HcCta c = p.ctas[cid];
    const NetZone z = p.zones[c.zone];
    const NetNode* __restrict__ nd = p.nodes + z.node0;
    const double2* __restrict__ wn = p.wn + z.node0;
    const int* __restrict__ lv = p.levels + z.lvl0;
    const int* __restrict__ rl = p.res + z.res0;
    const double* __restrict__ cumr = p.cumr + z.out_row;
    const int lg = c.lg, G = 1 << lg, T = p.T;
    const int items = z.n_nodes << lg;
    double* st = c.gstate < 0 ? hc_smem : p.gstate + c.gstate;
    double* th = st + items;
    const int g = threadIdx.x & (G - 1);        // this thread's step, the same in every loop below
    const int t = c.t0 + g;
    const bool on = t < T;
    const bool rated = p.scale != nullptr;
    double um = INFINITY;                       // uniform headroom of step t over this thread's nodes
    unsigned long long win = 0, open = 0, thermal = 0;

    if (on)
        for (int k = threadIdx.x; k < items; k += blockDim.x) {
            const NetNode n = nd[k >> lg];
            const double* Pt = p.P + (size_t)z.home_row * T + t;
            double f = 0.0;
            for (int e = 0; e < n.nres; ++e) f = __dadd_rn(f, Pt[(size_t)rl[n.res0 + e] * T]);
            st[k] = f;
        }
    __syncthreads();
    // leaves -> root: F, and the thermal terms of the rated edges
    for (int L = z.depth - 1; L >= 0; --L) {
        const int b = lv[L], w = lv[L + 1] - b;
        if (on)
            for (int k = threadIdx.x; k < (w << lg); k += blockDim.x) {
                const int q = b + (k >> lg);
                const NetNode n = nd[q];
                double f = st[(q << lg) + g];
                for (int e = 0; e < n.nchild; ++e) f = __dadd_rn(f, st[((n.child0 + e) << lg) + g]);
                st[(q << lg) + g] = f;
                if (rated) {
                    const double s = fabs(p.scale[z.out_row + n.node]);
                    double x = INFINITY;
                    if (s != 0.0) {
                        const double room = __dsub_rn(1.0, __dmul_rn(s, f));
                        x = __ddiv_rn(room, s);
                        const double na = wn[q].y;
                        if (na > 0.0) um = fmin(um, __ddiv_rn(room, __dmul_rn(s, na)));
                    }
                    th[(q << lg) + g] = x;
                }
            }
        __syncthreads();
    }
    // root -> leaves: D in place of F
    for (int L = 0; L < z.depth; ++L) {
        const int b = lv[L], w = lv[L + 1] - b;
        if (on)
            for (int k = threadIdx.x; k < (w << lg); k += blockDim.x) {
                const int q = b + (k >> lg);
                const NetNode n = nd[q];
                const double dp = n.parent < 0 ? 0.0 : st[(n.parent << lg) + g];
                st[(q << lg) + g] = __dadd_rn(dp, __dmul_rn(2.0 * n.r, st[(q << lg) + g]));
            }
        __syncthreads();
    }
    // leaves -> root: M, the smallest slack of the subtree, in place of D
    for (int L = z.depth - 1; L >= 0; --L) {
        const int b = lv[L], w = lv[L + 1] - b;
        if (on)
            for (int k = threadIdx.x; k < (w << lg); k += blockDim.x) {
                const int q = b + (k >> lg);
                const NetNode n = nd[q];
                double m = INFINITY;
                if (n.nres > 0) {
                    m = __dsub_rn(p.ur, st[(q << lg) + g]);
                    const double wq = wn[q].x;
                    if (wq > 0.0) um = fmin(um, __ddiv_rn(m, wq));
                }
                for (int e = 0; e < n.nchild; ++e) m = fmin(m, st[((n.child0 + e) << lg) + g]);
                st[(q << lg) + g] = m;
            }
        __syncthreads();
    }
    // root -> leaves: the running minima V (in place of M) and L (in place of th), and the residences' capacities
    for (int L = 0; L < z.depth; ++L) {
        const int b = lv[L], w = lv[L + 1] - b;
        if (on)
            for (int k = threadIdx.x; k < (w << lg); k += blockDim.x) {
                const int q = b + (k >> lg);
                const NetNode n = nd[q];
                const double d = 2.0 * cumr[n.node];
                double v = d > 0.0 ? __ddiv_rn(st[(q << lg) + g], d) : INFINITY;
                double l = rated ? th[(q << lg) + g] : INFINITY;
                if (n.parent >= 0) {
                    v = fmin(v, st[(n.parent << lg) + g]);
                    if (rated) l = fmin(l, th[(n.parent << lg) + g]);
                }
                st[(q << lg) + g] = v;
                if (rated) th[(q << lg) + g] = l;
                if (n.nres > 0) {
                    const double m = fmin(v, l);
                    const double cap = m > 0.0 ? m : 0.0;
                    if (l < v) thermal += (unsigned long long)n.nres;
                    for (int e = 0; e < n.nres; ++e) {
                        const int64_t hr = z.home_row + rl[n.res0 + e];
                        if (p.cap) p.cap[hr * T + t] = cap;
                        if (p.has_ev[hr] && t >= p.start[hr] && t < p.end[hr]) {
                            ++win;
                            if (cap >= p.rating[hr]) ++open;
                        }
                    }
                }
            }
        __syncthreads();
    }
    // the uniform headroom of every step: lanes g, g + G, ... of a warp, then the warps
    for (int o = 16; o >= G; o >>= 1) um = fmin(um, __shfl_xor_sync(0xffffffffu, um, o));
    win = hc_sum(win);
    open = hc_sum(open);
    thermal = hc_sum(thermal);
    double(*um_warp)[32] = reinterpret_cast<double(*)[32]>(hc_smem);       // the state's last reads were before the
    unsigned long long(*cnt_warp)[3] = reinterpret_cast<unsigned long long(*)[3]>(hc_smem + kHcWarps * 32);  // barrier
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane < G) um_warp[warp][lane] = um;
    if (lane == 0) {
        cnt_warp[warp][0] = win;
        cnt_warp[warp][1] = open;
        cnt_warp[warp][2] = thermal;
    }
    __syncthreads();
    if (p.uniform && threadIdx.x < G && c.t0 + (int)threadIdx.x < T) {
        double m = um_warp[0][threadIdx.x];
        for (int w = 1; w < kHcWarps; ++w) m = fmin(m, um_warp[w][threadIdx.x]);
        p.uniform[(int64_t)c.zone * T + c.t0 + threadIdx.x] = m > 0.0 ? m : 0.0;
    }
    if (threadIdx.x < 3) {
        unsigned long long a = 0;
        for (int w = 0; w < kHcWarps; ++w) a += cnt_warp[w][threadIdx.x];
        p.part[3 * (int64_t)cid + threadIdx.x] = a;
    }
}

// One thread per zone: the counts of the zone's CTAs, in CTA order.
__global__ void hosting_reduce_kernel(const unsigned long long* __restrict__ part, const int* __restrict__ zone_cta,
                                      int n_zones, int64_t* __restrict__ counts) {
    const int z = blockIdx.x * blockDim.x + threadIdx.x;
    if (z >= n_zones) return;
    unsigned long long a[3] = {0, 0, 0};
    for (int c = zone_cta[z]; c < zone_cta[z + 1]; ++c)
        for (int k = 0; k < 3; ++k) a[k] += part[3 * (int64_t)c + k];
    for (int k = 0; k < 3; ++k) counts[3 * (int64_t)z + k] = (int64_t)a[k];
}

void hc_prepare(const NetHost& h, int T, HcHost& o) {
    std::vector<int> lists[3];
    o = HcHost();
    o.zone_cta.assign(1, 0);
    o.wn.resize(h.nodes.size());
    for (size_t zi = 0; zi < h.zones.size(); ++zi) {
        const NetZone& z = h.zones[zi];
        // W and N of every node: the drop and the flow of 1 kW at every residence, with the network check's recurrences
        double2* wn = o.wn.data() + z.node0;
        const NetNode* nd = h.nodes.data() + z.node0;
        for (int q = 0; q < z.n_nodes; ++q) wn[q] = make_double2(0.0, 0.0);
        for (int q = z.n_nodes - 1; q >= 0; --q) {
            wn[q].y += (double)nd[q].nres;
            if (nd[q].parent >= 0) wn[nd[q].parent].y += wn[q].y;
        }
        for (int q = 0; q < z.n_nodes; ++q) {
            const double dp = nd[q].parent < 0 ? 0.0 : wn[nd[q].parent].x;
            const volatile double a = (2.0 * nd[q].r) * wn[q].y;     // two roundings, as on the device
            wn[q].x = dp + a;
        }
        const size_t one = 2 * (size_t)z.n_nodes * sizeof(double);
        int cls = 0;
        const int lg = net_zone_lg(one, T, &cls), G = 1 << lg;
        for (int t0 = 0; t0 < T; t0 += G) {
            HcCta c{(int)zi, t0, lg, 0, -1};
            if (cls == 2) {
                c.gstate = o.gstate_doubles;
                o.gstate_doubles += 2 * (int64_t)z.n_nodes;
            } else {
                o.class_smem[cls] = std::max(o.class_smem[cls], one * G);
            }
            lists[cls].push_back((int)o.ctas.size());
            o.ctas.push_back(c);
        }
        o.zone_cta.push_back((int)o.ctas.size());
    }
    for (int s = 0; s < 3; ++s) {
        o.class_off[s] = (int)o.lists.size();
        o.lists.insert(o.lists.end(), lists[s].begin(), lists[s].end());
    }
    o.class_off[3] = (int)o.lists.size();
    for (int s = 0; s < 3; ++s) o.class_smem[s] = std::max(o.class_smem[s], kHcScratch);
}

cudaError_t launch_hosting(const HcParams& P, const int* d_list, int n_ctas, size_t smem, cudaStream_t s) {
    if (n_ctas == 0) return cudaSuccess;
    // always the same value: solvers of one device may launch from several host threads at once
    cudaError_t e = cudaFuncSetAttribute(hosting_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kNetSmemMax);
    if (e != cudaSuccess) return e;
    hosting_kernel<<<n_ctas, kHcThreads, smem, s>>>(P, d_list);
    return cudaGetLastError();
}

cudaError_t launch_hosting_reduce(const unsigned long long* part, const int* zone_cta, int n_zones, int64_t* counts,
                                  cudaStream_t s) {
    if (n_zones == 0) return cudaSuccess;
    hosting_reduce_kernel<<<(n_zones + 255) / 256, 256, 0, s>>>(part, zone_cta, n_zones, counts);
    return cudaGetLastError();
}

}  // namespace revs
