// Voltage SCREENING contraction  V~ = R * G  in BF16 on the tensor cores, FP32 accumulate.
//
// Inside the ADMM loop the operator's LinDistFlow check (R_res @ g of Utility.network,
// lpsolver.py:183-194) only has to answer "which rows can violate v <= u?".  All terms of
// R g are non-negative, so a low-precision product has a rigorous RELATIVE error bound:
//     R <= R~ / (1 - 2^-8),  g <= g~ / (1 - 2^-8)   (BF16 keeps 8 significant bits: round to nearest loses up
//                                                   to 2^-8, the FP64 -> FP32 -> BF16 double rounding included)
//     FP32 accumulation of K exact BF16xBF16 products: v~ >= (1 - 2 K 2^-24) * exact sum (truncating
//     accumulator; measured on the B200 for both screening kernels: tests/test_gpu_screening.py)
//  => v <= v~ / ((1 - 2^-8)^2 (1 - 2^-9)) = 1.00983 v~ for K <= kScreenMaxN = 16384  (kScreenUp = 1.0099).
// Operands just below a rounding midpoint reach v = 1.0078 v~ at every K.
// Rows with v~ <= (1 - kScreenMargin) u are therefore PROVEN feasible ((1 - kScreenMargin) kScreenUp < 1);
// only the remaining
// candidates are re-evaluated exactly in FP64 (utility_qp.cu: exact_voltages), so the KKT
// test and the results are those of the FP64 path -- "BF16 with refinement".  The screening
// pass reads the sensitivity blocks at 2 bytes per entry instead of 8 and runs at the BF16
// tensor rate, ~10x less time than the FP64 DMMA contraction it replaces in the loop.
//
// Kernel: CTA tile 128 (rows) x 96 (hours) x 32 (k), 8 warps (4x2), mma.sync.m16n8k16.bf16
// with ldmatrix operand fetch from a 4-stage cp.async ring (72 KB, 3 CTAs per SM); rows of
// the shared tiles are padded to 40 elements (80 B) so that every ldmatrix phase is
// bank-conflict free.
// Columns whose QP has converged are skipped exactly like in contract_f64.cu.
#include <cuda_bf16.h>

#include "kernels.cuh"

namespace revs {

namespace {

constexpr int kSBM = 128, kSBN = 96, kSBK = 32, kSStages = 4;
constexpr int kSLd = kSBK + 8;            // padded row, in bf16 elements
constexpr int kSThreads = 256;
constexpr int kSWarpsM = 4, kSWarpsN = 2;
constexpr int kSMT = kSBM / kSWarpsM / 16;   // 2 m16 tiles per warp
constexpr int kSNT = kSBN / kSWarpsN / 8;    // 6 n8 tiles per warp
constexpr size_t kSSmem = (size_t)kSStages * (kSBM + kSBN) * kSLd * sizeof(__nv_bfloat16);

__device__ __forceinline__ void cp16(void* smem, const void* gmem, bool valid) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void ldsm_x4(unsigned& r0, unsigned& r1, unsigned& r2, unsigned& r3, const void* p) {
    unsigned s = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(s));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__global__ void __launch_bounds__(kSThreads, 3)
screen_bf16_kernel(const ScreenProblem* __restrict__ problems, const ContractTile* __restrict__ tiles, int T, double thr) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem_raw);          // [stages][BM][kSLd]
    __nv_bfloat16* sB = sA + (size_t)kSStages * kSBM * kSLd;                 // [stages][BN][kSLd]

    const ContractTile tile = tiles[blockIdx.x];
    const ScreenProblem pb = problems[tile.problem];
    const int m0 = tile.row0, n0 = blockIdx.y * kSBN;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp % kSWarpsM) * (kSBM / kSWarpsM);
    const int wn = (warp / kSWarpsM) * (kSBN / kSWarpsN);
    const int nk = (pb.K + kSBK - 1) / kSBK;

    unsigned act = 0xffffffffu;
    if (pb.col_status) {
        act = 0u;
#pragma unroll
        for (int j = 0; j < kSNT; ++j) {
            const int colj = n0 + wn + j * 8 + (lane & 7);
            const bool on = colj < T && pb.col_status[colj] == 0;
            if (__any_sync(0xffffffffu, on)) act |= 1u << j;
        }
        if (__syncthreads_or(act != 0u) == 0) return;
    }

    auto load_stage = [&](int stage, int kt) {
        const int k0 = kt * kSBK;
        __nv_bfloat16* a = sA + (size_t)stage * kSBM * kSLd;
        __nv_bfloat16* b = sB + (size_t)stage * kSBN * kSLd;
        for (int c = tid; c < kSBM * (kSBK / 8); c += kSThreads) {
            const int r = c / (kSBK / 8), q = c % (kSBK / 8);
            const bool ok = (m0 + r) < pb.M && (k0 + 8 * q) < pb.K;
            const __nv_bfloat16* src = reinterpret_cast<const __nv_bfloat16*>(pb.A_) + (size_t)(ok ? m0 + r : 0) * pb.lda + (ok ? k0 + 8 * q : 0);
            cp16(a + r * kSLd + 8 * q, src, ok);
        }
        for (int c = tid; c < kSBN * (kSBK / 8); c += kSThreads) {
            const int r = c / (kSBK / 8), q = c % (kSBK / 8);
            const bool ok = (n0 + r) < T && (k0 + 8 * q) < pb.K;
            const __nv_bfloat16* src = reinterpret_cast<const __nv_bfloat16*>(pb.Bt_) + (size_t)(ok ? n0 + r : 0) * pb.ldb + (ok ? k0 + 8 * q : 0);
            cp16(b + r * kSLd + 8 * q, src, ok);
        }
    };

    float acc[kSMT][kSNT][4];
#pragma unroll
    for (int i = 0; i < kSMT; ++i)
#pragma unroll
        for (int j = 0; j < kSNT; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.f;

#pragma unroll
    for (int s = 0; s < kSStages - 1; ++s) {
        if (s < nk) load_stage(s, s);
        asm volatile("cp.async.commit_group;\n" ::);
    }
    for (int kt = 0; kt < nk; ++kt) {
        asm volatile("cp.async.wait_group %0;\n" ::"n"(kSStages - 2));
        __syncthreads();
        {
            const int nxt = kt + kSStages - 1;
            if (nxt < nk) load_stage(nxt % kSStages, nxt);
            asm volatile("cp.async.commit_group;\n" ::);
        }
        const __nv_bfloat16* a = sA + (size_t)(kt % kSStages) * kSBM * kSLd;
        const __nv_bfloat16* b = sB + (size_t)(kt % kSStages) * kSBN * kSLd;
#pragma unroll
        for (int kk = 0; kk < kSBK; kk += 16) {
            unsigned af[kSMT][4];
#pragma unroll
            for (int i = 0; i < kSMT; ++i) {
                // x4: matrices (rows 0-7,k 0-7), (rows 8-15,k 0-7), (rows 0-7,k 8-15), (rows 8-15,k 8-15)
                const int r = wm + i * 16 + (lane & 15), c = kk + ((lane >> 4) << 3);
                ldsm_x4(af[i][0], af[i][1], af[i][2], af[i][3], a + r * kSLd + c);
            }
#pragma unroll
            for (int jp = 0; jp < kSNT; jp += 2) {
                if (!(act & (3u << jp))) continue;
                // x4 over two n8 tiles: (n 0-7,k 0-7), (n 0-7,k 8-15), (n 8-15,k 0-7), (n 8-15,k 8-15)
                unsigned b0, b1, b2, b3;
                const int r = wn + jp * 8 + (lane & 7) + ((lane >> 4) << 3), c = kk + (((lane >> 3) & 1) << 3);
                ldsm_x4(b0, b1, b2, b3, b + r * kSLd + c);
#pragma unroll
                for (int i = 0; i < kSMT; ++i) {
                    if (act & (1u << jp)) mma_bf16(acc[i][jp], af[i], b0, b1);
                    if (act & (2u << jp)) mma_bf16(acc[i][jp + 1], af[i], b2, b3);
                }
            }
        }
    }
    asm volatile("cp.async.wait_group 0;\n" ::);

    // epilogue: c0,c1 -> (row g, cols 2t,2t+1); c2,c3 -> (row g+8, ...); time-major fp32
    const int g8 = lane >> 2, t4 = lane & 3;
#pragma unroll
    for (int i = 0; i < kSMT; ++i)
#pragma unroll
        for (int j = 0; j < kSNT; ++j) {
            if (!(act & (1u << j))) continue;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int row = m0 + wm + i * 16 + g8 + ((e >> 1) << 3);
                const int colj = n0 + wn + j * 8 + 2 * t4 + (e & 1);
                if (row < pb.M && colj < T) {
                    pb.out[(size_t)colj * pb.ldo + row] = acc[i][j][e];
                    if (pb.col_cand && (double)acc[i][j][e] > thr) pb.col_cand[colj] = 1;   // the column needs the QP kernel
                }
            }
        }
}

__global__ void to_bf16_kernel(const double* __restrict__ in, __nv_bfloat16* __restrict__ out, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = __float2bfloat16_rn((float)in[i]);
}

}  // namespace

int screen_tile_rows() { return kSBM; }

cudaError_t launch_to_bf16(const double* in, void* out, size_t n, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    to_bf16_kernel<<<(unsigned)blocks, 256, 0, s>>>(in, reinterpret_cast<__nv_bfloat16*>(out), n);
    return cudaGetLastError();
}

cudaError_t screen_prepare() {
    static std::atomic<unsigned long long> attr_devices{0};
    if (first_use_on_device(attr_devices))
        return cudaFuncSetAttribute(screen_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSSmem);
    return cudaSuccess;
}

cudaError_t launch_screen(const ScreenProblem* d_problems, const ContractTile* d_tiles, int n_tiles, int T, double thr,
                          cudaStream_t stream) {
    if (n_tiles == 0) return cudaSuccess;
    cudaError_t pe = screen_prepare();
    if (pe != cudaSuccess) return pe;
    screen_bf16_kernel<<<dim3(n_tiles, (T + kSBN - 1) / kSBN), kSThreads, kSSmem, stream>>>(d_problems, d_tiles, T, thr);
    return cudaGetLastError();
}

}  // namespace revs
