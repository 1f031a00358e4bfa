// Network check of a whole population (revs_network_check): LinDistFlow voltages and line flows of every node, every
// zone and every step from the residences' schedule, without a sensitivity matrix.
//
// Per zone and step (nodes topological, r_i = cumr[i] - cumr[parent[i]]):
//     F_i = inj_i + sum_{children c} F_c      leaves -> root   (flow on the edge above i, inj = the node's residences)
//     D_i = D_parent(i) + 2 r_i F_i           root -> leaves   (D = R P at node i, the squared-voltage drop)
// which is what revs_reliability computes by contracting dense path-indicator blocks (feeder_build.cu), in
// O(nodes x T) instead of O(nodes x residences x depth).
//
// One CTA per (zone, group of G steps).  The zone's nodes are renumbered breadth-first on the host (net_add_zone), so
// the children of a node are contiguous in the next level, and the CTA walks the levels: threads over (node of the
// level, step), one barrier per level, depth-many barriers per pass.  The per-node state of a step is one double
// (F, then D in place), [nodes][G] in shared memory; G is chosen per zone from its node count alone, so a zone's
// result does not depend on the zones that share the solver.  A zone whose one-step state does not fit in shared
// memory runs the same code on a global (L2-resident) scratch.
//
// Sums are taken in a fixed order (residences by home index, then children by node index) with explicit
// round-to-nearest adds and multiplies, so the outputs equal the numpy model of tests/network_ref.py bit for bit.
// Maxima are reduced under a total order (value, then lowest zone / index / step), counts are integers: the
// summary is the same for any CTA schedule.
#include <algorithm>
#include <cmath>

#include "kernels.cuh"

namespace revs {

namespace {

constexpr int kNetThreads = 256;
constexpr int kNetWarps = kNetThreads / 32;

__device__ __forceinline__ bool net_better(const NetArg& a, const NetArg& b) {
    return a.v > b.v || (a.v == b.v && (a.zone < b.zone || (a.zone == b.zone && a.loc < b.loc)));
}

__device__ __forceinline__ void net_take(NetArg& a, double v, int zone, int64_t loc) {
    const NetArg b{v, zone, 0, loc};
    if (net_better(b, a)) a = b;
}

__device__ __forceinline__ NetArg net_shfl(const NetArg& a, int o) {
    NetArg b;
    b.v = __shfl_xor_sync(0xffffffffu, a.v, o);
    b.zone = __shfl_xor_sync(0xffffffffu, a.zone, o);
    b.pad_ = 0;
    b.loc = __shfl_xor_sync(0xffffffffu, a.loc, o);
    return b;
}

__device__ __forceinline__ unsigned long long net_sum(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ NetArg net_none() { return NetArg{-INFINITY, 0x7fffffff, 0, INT64_MAX}; }

// block-wide combination of the per-thread partials; the result is valid in thread 0
__device__ NetPartial net_block_reduce(NetPartial m) {
    __shared__ NetPartial warp_part[kNetWarps];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        NetArg b = net_shfl(m.drop, o);
        if (net_better(b, m.drop)) m.drop = b;
        b = net_shfl(m.exc, o);
        if (net_better(b, m.exc)) m.exc = b;
        b = net_shfl(m.load, o);
        if (net_better(b, m.load)) m.load = b;
    }
    m.rows = net_sum(m.rows);
    m.low = net_sum(m.low);
    m.over = net_sum(m.over);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) warp_part[warp] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
            const NetPartial& x = warp_part[w];
            if (net_better(x.drop, m.drop)) m.drop = x.drop;
            if (net_better(x.exc, m.exc)) m.exc = x.exc;
            if (net_better(x.load, m.load)) m.load = x.load;
            m.rows += x.rows;
            m.low += x.low;
            m.over += x.over;
        }
    }
    return m;
}

}  // namespace

__global__ void __launch_bounds__(kNetThreads) network_check_kernel(NetParams p, const int* __restrict__ list) {
    extern __shared__ double net_smem[];
    const int cid = list[blockIdx.x];
    const NetCta c = p.ctas[cid];
    const NetZone z = p.zones[c.zone];
    const NetNode* __restrict__ nd = p.nodes + z.node0;
    const int* __restrict__ lv = p.levels + z.lvl0;
    const int* __restrict__ rl = p.res + z.res0;
    double* st = c.gstate < 0 ? net_smem : p.gstate + c.gstate;
    const int lg = z.lg, G = 1 << lg, T = p.T;
    const int ng = min(G, T - c.t0);           // steps of this CTA
    const int items = z.n_nodes << lg;

    // injections of all nodes at once (no dependence between nodes)
    for (int k = threadIdx.x; k < items; k += blockDim.x) {
        const int g = k & (G - 1);
        if (g >= ng) continue;
        const NetNode n = nd[k >> lg];
        const double* Pt = p.P + (size_t)z.home_row * T + c.t0 + g;
        double f = 0.0;
        for (int e = 0; e < n.nres; ++e) f = __dadd_rn(f, Pt[(size_t)rl[n.res0 + e] * T]);
        st[k] = f;
    }
    __syncthreads();

    NetPartial m;
    m.drop = m.exc = m.load = net_none();
    m.rows = m.low = m.over = 0;
    // leaves -> root: F
    for (int L = z.depth - 1; L >= 0; --L) {
        const int b = lv[L], w = lv[L + 1] - b;
        for (int k = threadIdx.x; k < (w << lg); k += blockDim.x) {
            const int g = k & (G - 1);
            if (g >= ng) continue;
            const int q = b + (k >> lg);
            const NetNode n = nd[q];
            double f = st[(q << lg) + g];
            for (int e = 0; e < n.nchild; ++e) f = __dadd_rn(f, st[((n.child0 + e) << lg) + g]);
            st[(q << lg) + g] = f;
            const int t = c.t0 + g;
            const int64_t row = z.out_row + n.node;
            const double lf = p.scale ? __dmul_rn(p.scale[row], f) : f;
            if (p.loading) p.loading[row * T + t] = lf;
            const double a = fabs(lf);
            net_take(m.load, a, c.zone, (int64_t)n.node * T + t);
            if (p.scale && a > 1.0) ++m.over;
        }
        __syncthreads();
    }
    // root -> leaves: D (in place of F)
    for (int L = 0; L < z.depth; ++L) {
        const int b = lv[L], w = lv[L + 1] - b;
        for (int k = threadIdx.x; k < (w << lg); k += blockDim.x) {
            const int g = k & (G - 1);
            if (g >= ng) continue;
            const int q = b + (k >> lg);
            const NetNode n = nd[q];
            const double dp = n.parent < 0 ? 0.0 : st[(n.parent << lg) + g];
            const double d = __dadd_rn(dp, __dmul_rn(2.0 * n.r, st[(q << lg) + g]));
            st[(q << lg) + g] = d;
            const int t = c.t0 + g;
            const int64_t row = z.out_row + n.node;
            if (p.voltage) p.voltage[row * T + t] = sqrt(p.v2 - d);
            net_take(m.drop, d, c.zone, (int64_t)n.node * T + t);
            if (d > p.low) ++m.low;
            if (n.nres > 0) {
                if (p.drop) {
                    double* dt = p.drop + z.home_row * T + (int64_t)t * z.n_res;
                    for (int e = 0; e < n.nres; ++e) dt[rl[n.res0 + e]] = d;
                }
                const double x = d - p.u;
                net_take(m.exc, x, c.zone, (int64_t)rl[n.res0] * T + t);     // first (lowest) residence of the node
                if (x > p.row_tol) m.rows += (unsigned long long)n.nres;
            }
        }
        __syncthreads();
    }
    m = net_block_reduce(m);
    if (threadIdx.x == 0) p.part[cid] = m;
}

// One CTA: the CTAs of every zone in order -> zone_worst, then all zones -> the summary.
__global__ void __launch_bounds__(kNetThreads) network_reduce_kernel(const NetPartial* __restrict__ part,
                                                                       const int* __restrict__ zone_cta, int n_zones,
                                                                       double* __restrict__ zone_worst,
                                                                       NetPartial* __restrict__ out) {
    NetPartial m;
    m.drop = m.exc = m.load = net_none();
    m.rows = m.low = m.over = 0;
    for (int z = threadIdx.x; z < n_zones; z += blockDim.x) {
        NetPartial a;
        a.drop = a.exc = a.load = net_none();
        for (int c = zone_cta[z]; c < zone_cta[z + 1]; ++c) {
            const NetPartial& x = part[c];
            if (net_better(x.drop, a.drop)) a.drop = x.drop;
            if (net_better(x.exc, a.exc)) a.exc = x.exc;
            if (net_better(x.load, a.load)) a.load = x.load;
            m.rows += x.rows;
            m.low += x.low;
            m.over += x.over;
        }
        zone_worst[3 * (size_t)z + 0] = a.drop.v;
        zone_worst[3 * (size_t)z + 1] = a.exc.v;
        zone_worst[3 * (size_t)z + 2] = a.load.v;
        if (net_better(a.drop, m.drop)) m.drop = a.drop;
        if (net_better(a.exc, m.exc)) m.exc = a.exc;
        if (net_better(a.load, m.load)) m.load = a.load;
    }
    m = net_block_reduce(m);
    if (threadIdx.x == 0) *out = m;
}

void net_add_zone(NetHost& h, int n_nodes, const int* parent, const double* cumr, int n_res, const int* res_node,
                  int64_t home_row) {
    BfsTree B;
    bfs_tree(n_nodes, parent, n_res, res_node, B);
    NetZone z{};
    z.node0 = (int64_t)h.nodes.size();
    z.lvl0 = (int64_t)h.levels.size();
    z.res0 = (int64_t)h.res.size();
    z.home_row = home_row;
    z.out_row = h.total_nodes;
    z.n_nodes = n_nodes;
    z.n_res = n_res;
    z.depth = (int)B.lvl.size() - 1;
    h.levels.insert(h.levels.end(), B.lvl.begin(), B.lvl.end());
    h.res.insert(h.res.end(), B.res.begin(), B.res.end());
    for (int q = 0; q < n_nodes; ++q) {
        const int i = B.order[q], pa = parent[i];
        NetNode nd{};
        nd.r = pa < 0 ? cumr[i] : cumr[i] - cumr[pa];
        nd.node = i;
        nd.parent = B.parent[q];
        nd.child0 = B.child0[q];
        nd.nchild = B.nchild[q];
        nd.res0 = B.res0[q];
        nd.nres = B.nres[q];
        h.nodes.push_back(nd);
    }
    h.zones.push_back(z);
    h.total_nodes += n_nodes;
}

int net_zone_lg(size_t one, int T, int* cls) {
    int G = 1;
    while (G < T && G < kNetMaxSteps) G <<= 1;
    *cls = 0;
    while (G > 1 && one * G > kNetSmemSmall) G >>= 1;
    if (one * G > kNetSmemSmall) *cls = one <= kNetSmemMax ? 1 : 2;
    int lg = 0;
    while ((1 << lg) < G) ++lg;
    return lg;
}

void net_finish(NetHost& h, int T) {
    std::vector<int> lists[3];
    h.zone_cta.assign(1, 0);
    h.ctas.clear();
    h.gstate_doubles = 0;
    for (size_t s = 0; s < 3; ++s) h.class_smem[s] = 0;
    for (size_t zi = 0; zi < h.zones.size(); ++zi) {
        NetZone& z = h.zones[zi];
        const size_t one = (size_t)z.n_nodes * sizeof(double);
        int cls = 0;
        z.lg = net_zone_lg(one, T, &cls);
        const int G = 1 << z.lg;
        for (int t0 = 0; t0 < T; t0 += G) {
            NetCta c{(int)zi, t0, -1};
            if (cls == 2) {
                c.gstate = h.gstate_doubles;
                h.gstate_doubles += z.n_nodes;
            } else {
                h.class_smem[cls] = std::max(h.class_smem[cls], one * G);
            }
            lists[cls].push_back((int)h.ctas.size());
            h.ctas.push_back(c);
        }
        h.zone_cta.push_back((int)h.ctas.size());
    }
    h.lists.clear();
    for (int s = 0; s < 3; ++s) {
        h.class_off[s] = (int)h.lists.size();
        h.lists.insert(h.lists.end(), lists[s].begin(), lists[s].end());
    }
    h.class_off[3] = (int)h.lists.size();
}

cudaError_t launch_network_check(const NetParams& P, const int* d_list, int n_ctas, size_t smem, cudaStream_t s) {
    if (n_ctas == 0) return cudaSuccess;
    // always the same value: solvers of one device may launch from several host threads at once
    cudaError_t e = cudaFuncSetAttribute(network_check_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kNetSmemMax);
    if (e != cudaSuccess) return e;
    network_check_kernel<<<n_ctas, kNetThreads, smem, s>>>(P, d_list);
    return cudaGetLastError();
}

cudaError_t launch_network_reduce(const NetPartial* part, const int* zone_cta, int n_zones, double* zone_worst,
                                  NetPartial* out, cudaStream_t s) {
    network_reduce_kernel<<<1, kNetThreads, 0, s>>>(part, zone_cta, n_zones, zone_worst, out);
    return cudaGetLastError();
}

}  // namespace revs
