// Sensitivity matrices of a radial feeder, built on the device from the tree itself.
//
// Reference: compute_Rmat (lpsolver.py:17-26) forms R = 2 F D F^T by inverting the reduced
// incidence matrix with numpy; compute_flows (drawing.py:29-59) inverts it again for the
// flow sensitivities.  For a radial feeder both inverses are path indicators, so
//     R[a][b]   = 2 * (resistance of the common part of the root paths of a and b)
//     A_inv[e][b] = +-1 iff edge e lies on the root path of b
// and each entry is one walk up the tree.  Nodes are topologically numbered
// (parent[i] < i, -1 = substation), so the lowest common ancestor is found by lifting
// whichever index is larger.
#include "kernels.cuh"

namespace revs {

// out[m*ld + j] for m < n_rows, j < n_res.  row_node == nullptr means rows are the residences.
__global__ void sens_voltage_kernel(const int* __restrict__ parent, const double* __restrict__ cumr,
                                    const int* __restrict__ row_node, const int* __restrict__ res_node,
                                    int n_rows, int n_res, double* __restrict__ out, int ld) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_res) return;
    for (int m = blockIdx.y; m < n_rows; m += gridDim.y) {
        int a = row_node ? row_node[m] : res_node[m];
        int b = res_node[j];
        while (a != b) {
            if (a > b) a = parent[a];
            else b = parent[b];
        }
        out[(size_t)m * ld + j] = a < 0 ? 0.0 : 2.0 * cumr[a];
    }
}

// All residence blocks of a batch of feeders in one launch (blockIdx.z = feeder).
__global__ void sens_voltage_batched_kernel(const FeederDev* __restrict__ feeders, const int64_t* __restrict__ node_off,
                                            const int* __restrict__ parent, const double* __restrict__ cumr,
                                            const int* __restrict__ res_node, double* __restrict__ Rpool) {
    const FeederDev fd = feeders[blockIdx.z];
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= fd.n || fd.roff < 0) return;          // roff < 0: zone of the tree-Newton path, no dense block
    const int* par = parent + node_off[blockIdx.z];
    const double* cr = cumr + node_off[blockIdx.z];
    const int* res = res_node + fd.off;
    const int bj = res[j];
    for (int m = blockIdx.y; m < fd.n; m += gridDim.y) {
        int a = res[m], b = bj;
        while (a != b) {
            if (a > b) a = par[a];
            else b = par[b];
        }
        Rpool[fd.roff + (size_t)m * fd.np + j] = a < 0 ? 0.0 : 2.0 * cr[a];
    }
}

// out[m*ld + j] = 1 if the edge above node row_node[m] carries residence j.
__global__ void sens_flow_kernel(const int* __restrict__ parent, const int* __restrict__ row_node,
                                 const int* __restrict__ res_node, int n_rows, int n_res,
                                 double* __restrict__ out, int ld) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_res) return;
    for (int m = blockIdx.y; m < n_rows; m += gridDim.y) {
        const int e = row_node[m];
        int b = res_node[j];
        while (b > e) b = parent[b];
        out[(size_t)m * ld + j] = (b == e) ? 1.0 : 0.0;
    }
}

// home-major [n][T] -> time-major [T][ld]
__global__ void to_time_major_kernel(const double* __restrict__ in, int n, int T, double* __restrict__ out,
                                     int64_t ld) {
    __shared__ double tile[32][33];
    const int h0 = blockIdx.x * 32, t0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int h = h0 + r, t = t0 + threadIdx.x;
        tile[r][threadIdx.x] = (h < n && t < T) ? in[(size_t)h * T + t] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int t = t0 + r, h = h0 + threadIdx.x;
        if (t < T && h < n) out[(size_t)t * ld + h] = tile[threadIdx.x][r];
    }
}

// rn2[off + i] = sum_j R_f[i][j]^2 : curvature scale of the utility QP, one warp per row
__global__ void row_norms_kernel(const FeederDev* __restrict__ feeders, const double* __restrict__ Rpool,
                                 double* __restrict__ rn2, double* __restrict__ rmax) {
    const FeederDev fd = feeders[blockIdx.y];
    const int lane = threadIdx.x & 31;
    if (fd.roff < 0) return;
    for (int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < fd.n; i += gridDim.x * (blockDim.x >> 5)) {
        const double* row = Rpool + fd.roff + (size_t)i * fd.np;
        double acc = 0.0, mx = 0.0;
        for (int j = lane; j < fd.n; j += 32) { acc = fma(row[j], row[j], acc); mx = fmax(mx, row[j]); }
        acc = warp_sum(acc);
        mx = warp_max(mx);
        if (lane == 0) { rn2[fd.off + i] = acc; rmax[fd.off + i] = mx; }
    }
}

cudaError_t launch_row_norms(const FeederDev* feeders, int n_feeders, const double* Rpool, double* rn2, double* rmax,
                             cudaStream_t s) {
    row_norms_kernel<<<dim3(64, n_feeders), 256, 0, s>>>(feeders, Rpool, rn2, rmax);
    return cudaGetLastError();
}

cudaError_t launch_sens_voltage(const int* parent, const double* cumr, const int* row_node,
                                const int* res_node, int n_rows, int n_res, double* out, int ld,
                                cudaStream_t s) {
    if (n_rows == 0 || n_res == 0) return cudaSuccess;
    dim3 grid((n_res + 127) / 128, n_rows < 65535 ? n_rows : 65535);
    sens_voltage_kernel<<<grid, 128, 0, s>>>(parent, cumr, row_node, res_node, n_rows, n_res, out, ld);
    return cudaGetLastError();
}
cudaError_t launch_sens_voltage_batched(const FeederDev* feeders, int n_feeders, int max_n, const int64_t* node_off,
                                        const int* parent, const double* cumr, const int* res_node, double* Rpool,
                                        cudaStream_t s) {
    if (n_feeders == 0 || max_n == 0) return cudaSuccess;
    for (int f0 = 0; f0 < n_feeders; f0 += 65535) {
        const int nz = n_feeders - f0 < 65535 ? n_feeders - f0 : 65535;
        dim3 grid((max_n + 127) / 128, max_n < 256 ? max_n : 256, nz);
        sens_voltage_batched_kernel<<<grid, 128, 0, s>>>(feeders + f0, node_off + f0, parent, cumr, res_node, Rpool);
    }
    return cudaGetLastError();
}
cudaError_t launch_sens_flow(const int* parent, const int* row_node, const int* res_node, int n_rows,
                             int n_res, double* out, int ld, cudaStream_t s) {
    if (n_rows == 0 || n_res == 0) return cudaSuccess;
    dim3 grid((n_res + 127) / 128, n_rows < 65535 ? n_rows : 65535);
    sens_flow_kernel<<<grid, 128, 0, s>>>(parent, row_node, res_node, n_rows, n_res, out, ld);
    return cudaGetLastError();
}
// compact [H][w] <-> padded [Hp][w] home-major arrays (hmap[h] = padded row of compact home h)
__global__ void pack_rows_kernel(const double* __restrict__ src, double* __restrict__ dst, const int64_t* __restrict__ hmap,
                                 int64_t H, int w, int to_padded) {
    const int64_t total = H * w;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t h = i / w;
        const int k = (int)(i - h * w);
        const int64_t p = hmap[h] * w + k;
        if (to_padded) dst[p] = src[i];
        else dst[i] = src[p];
    }
}

cudaError_t launch_pack_rows(const double* src, double* dst, const int64_t* hmap, int64_t H, int w, int to_padded,
                             cudaStream_t s) {
    if (H == 0) return cudaSuccess;
    int64_t blocks = (H * w + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    pack_rows_kernel<<<(unsigned)blocks, 256, 0, s>>>(src, dst, hmap, H, w, to_padded);
    return cudaGetLastError();
}

// charging decisions as bit masks: bit (t & 63) of word t / 64 of compact home h is set when the charger runs in
// step t.  One warp per home, two ballots per 64-bit word.
__global__ void hour_mask_kernel(const double* __restrict__ p_ev, const int64_t* __restrict__ hmap, int64_t H, int T,
                                 int words, unsigned long long* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t h = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (h >= H) return;
    const double* row = p_ev + hmap[h] * T;
    for (int w = 0; w < words; ++w) {
        const int t0 = 64 * w + lane, t1 = t0 + 32;
        const unsigned lo = __ballot_sync(0xffffffffu, t0 < T && row[t0] > 0.0);
        const unsigned hi = __ballot_sync(0xffffffffu, t1 < T && row[t1] > 0.0);
        if (lane == 0) out[h * words + w] = (unsigned long long)lo | ((unsigned long long)hi << 32);
    }
}

cudaError_t launch_hour_mask(const double* p_ev, const int64_t* hmap, int64_t H, int T, unsigned long long* out, cudaStream_t s) {
    if (H == 0) return cudaSuccess;
    const int wpb = 8;
    hour_mask_kernel<<<(unsigned)((H + wpb - 1) / wpb), 32 * wpb, 0, s>>>(p_ev, hmap, H, T, (T + 63) / 64, out);
    return cudaGetLastError();
}

cudaError_t launch_to_time_major(const double* in, int n, int T, double* out, int64_t ld, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    dim3 grid((n + 31) / 32, (T + 31) / 32), block(32, 8);
    to_time_major_kernel<<<grid, block, 0, s>>>(in, n, T, out, ld);
    return cudaGetLastError();
}

void bfs_tree(int n_nodes, const int* parent, int n_res, const int* res_node, BfsTree& B) {
    const int n = n_nodes;
    // children and residences of every node, ascending
    std::vector<int> cofs(n + 1, 0), kids(n), rofs(n + 1, 0), homes(n_res);
    for (int i = 0; i < n; ++i)
        if (parent[i] >= 0) ++cofs[parent[i] + 1];
    for (int j = 0; j < n_res; ++j) ++rofs[res_node[j] + 1];
    for (int i = 0; i < n; ++i) { cofs[i + 1] += cofs[i]; rofs[i + 1] += rofs[i]; }
    {
        std::vector<int> fill(cofs.begin(), cofs.end() - 1);
        for (int i = 0; i < n; ++i)
            if (parent[i] >= 0) kids[fill[parent[i]]++] = i;
        std::vector<int> rf(rofs.begin(), rofs.end() - 1);
        for (int j = 0; j < n_res; ++j) homes[rf[res_node[j]]++] = j;
    }
    B.order.clear();
    B.order.reserve(n);
    for (int i = 0; i < n; ++i)
        if (parent[i] < 0) B.order.push_back(i);
    B.lvl.assign(1, 0);
    for (size_t lo = 0; lo < B.order.size();) {
        const size_t hi = B.order.size();
        B.lvl.push_back((int)hi);
        for (size_t q = lo; q < hi; ++q)
            for (int e = cofs[B.order[q]]; e < cofs[B.order[q] + 1]; ++e) B.order.push_back(kids[e]);
        lo = hi;
    }
    std::vector<int> pos(n);
    for (int q = 0; q < n; ++q) pos[B.order[q]] = q;
    B.parent.resize(n); B.child0.resize(n); B.nchild.resize(n); B.res0.resize(n); B.nres.resize(n);
    B.res.clear();
    B.res.reserve(n_res);
    for (int q = 0; q < n; ++q) {
        const int i = B.order[q];
        B.parent[q] = parent[i] < 0 ? -1 : pos[parent[i]];
        B.nchild[q] = cofs[i + 1] - cofs[i];
        B.child0[q] = B.nchild[q] ? pos[kids[cofs[i]]] : 0;
        B.res0[q] = (int)B.res.size();
        B.nres[q] = rofs[i + 1] - rofs[i];
        B.res.insert(B.res.end(), homes.begin() + rofs[i], homes.begin() + rofs[i + 1]);
    }
}

}  // namespace revs
