// Shared device-side definitions of the REVS ADMM path (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

namespace revs {

constexpr int kPad = 16;        // residences of a feeder are padded to a multiple of this
constexpr int kWMax = 128;      // largest working set of a (feeder,hour) utility QP column
constexpr int kAddMax = 32;     // violated voltage rows admitted per working-set round
constexpr int kWW = 16;         // working-set capacity of the warp-per-column QP kernel
constexpr int kQpClasses = 4;   // utility QP instantiations: 0 = warp kernel, 1..3 = CTA kernels by capacity
constexpr int kQpLists = 17;    // work lists: classes 1..3 at [1..3], the warp kernels' buckets at [4..7] (zones <= 128), [8..11] (<= 256)
                                // and [13..16] (<= 320), [12] = columns the one-row kernel passes on to the general warp kernel
constexpr int kListLeftover = 12;
constexpr int kListBig = 13;    // first bucket of the zones of 257..kWarpMaxN residences
constexpr int kWarpMaxN = 320;  // largest zone the warp-per-column QP kernel takes (the reference feeder's zones: 157..297)
__host__ __device__ constexpr int qp_class_cap(int cls) { return cls == 0 ? kWW : (cls == 1 ? 32 : (cls == 2 ? 64 : kWMax)); }

// One feeder of the batch as the kernels see it.
struct FeederDev {
    int n;            // residences
    int np;           // padded residences (multiple of kPad) == leading dim of R block
    int64_t off;      // first padded home index
    int64_t roff;     // offset (doubles) of the n_p x n_p block in the R pool; -1: no dense block (tree-Newton zone)
};

// Output layout / transform of the sensitivity contraction.
enum ContractOut : int {
    kOutTimeMajor = 0,   // out[t*ldo + m] = acc
    kOutNodeMajor = 1,   // out[m*ldo + t] = acc
    kOutVoltage = 2,     // out[m*ldo + t] = sqrt(v2 - acc)
    kOutScaled = 3       // out[m*ldo + t] = scale[m] * acc
};

// All-gather fused into the contraction epilogue (one feeder row-partitioned over the GPUs of a box): every output
// element is stored into the gather buffer of EVERY rank (peer-mapped memory, NVLink stores) at the rows this rank
// owns; the last CTA of the kernel then raises this rank's flag in every peer's buffer (system-scope release).
constexpr int kGatherMaxPeers = 16;
struct GatherDev {
    double* out[kGatherMaxPeers];                  // payload of every rank's gather buffer (out[rank] is local)
    unsigned long long* flag[kGatherMaxPeers];     // flag[r] + my rank: my arrival flag in rank r's buffer
    unsigned* ticket;                              // local CTA counter (zero before the launch)
    unsigned long long seq;                        // value of this exchange
    int world, rank;
    int row_base;                                  // first gathered row this rank owns
    int64_t ldo;                                   // leading dimension of the gathered output
};

// Batched contraction problem: C_f = A_f (M_f x K_f) * B_f^T (T x K_f).
struct ContractProblem {
    const double* A; int lda; int M; int K;
    const double* Bt; int64_t ldb;       // Bt[t*ldb + k]
    double* out; int64_t ldo;
    const double* scale;                 // per-row, kOutScaled only
    const int* col_status;               // optional [T]: columns with status != 0 are skipped
    const GatherDev* gather;             // optional: node-major outputs go to every rank's gather buffer instead of `out`
};

struct ContractTile { int problem; int row0; };

// Screening contraction (BF16 in, FP32 out, time-major): V~_f = A_f (M x K) * B_f^T (T x K).
struct ScreenProblem {
    const void* A_; int lda; int M; int K;      // __nv_bfloat16
    const void* Bt_; int64_t ldb;               // __nv_bfloat16, Bt[t*ldb + k]
    float* out; int64_t ldo;                    // out[t*ldo + m]
    const int* col_status;                      // optional [T]: columns with status != 0 are skipped
    int* col_cand;                              // optional [T]: set to 1 when any row of the column has v~ > thr
};

constexpr double kScreenMargin = 0.01;   // rows with v~ <= (1-margin) u are proven feasible (see screen_bf16.cu)
constexpr double kScreenUp = 1.0099;     // v <= kScreenUp * v~ for the BF16/FP32 product of non-negative terms, K <= kScreenMaxN
constexpr int kScreenMaxN = 16384;       // largest zone (K of the screening product) the bound above holds for
constexpr int kVerifyMaxN = 512;         // zones up to this size verify all voltage rows inside the QP kernels
constexpr int kQpBuckets = 4;            // work lists of the warp kernel: |W| >= 3, 2, 1, 0 (hardest first)

// Function attributes (dynamic shared-memory size, carve-out) are per device.  Returns true the first time it is
// called for `mask` on the current device, so a launcher sets its attributes once per device, from any host thread.
inline bool first_use_on_device(std::atomic<unsigned long long>& mask) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return true;
    const unsigned long long bit = 1ull << (dev & 63);
    return (mask.fetch_or(bit) & bit) == 0;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace revs
