// C ABI and device-side orchestration of the REVS ADMM path (see include/revs_admm.h).
//
// One revs_solver owns everything a batch of feeders needs on one B200: the dense
// sensitivity blocks (n_f^2 doubles per feeder, 128-byte aligned, residences padded to a
// multiple of 16 so every cp.async of the contraction is aligned), the home-major
// [Hp][T] arrays of the consumer side, the time-major [T][Hp] arrays of the operator
// side, the per-(feeder,hour) working sets and a small pinned block of counters that is
// the only thing the host reads while the loop runs.
//
// An ADMM iteration (lpsolver.py:254-287) is, on the device:
//   stream U:  utility_qp(init) -> { contract_f64 ; utility_qp(step) } until no column runs
//   stream H:  home_solve           (uses the PREVIOUS iterates, so it overlaps stream U)
//   stream U:  dual_update          (after both)
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <cstdlib>
#include <cmath>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/revs_admm.h"
#include "kernels.cuh"

using namespace revs;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(x)                                                                               \
    do {                                                                                    \
        cudaError_t e_ = (x);                                                               \
        if (e_ != cudaSuccess)                                                              \
            return fail(REVS_ERR_CUDA, "%s failed: %s (%s:%d)", #x, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                \
    } while (0)

constexpr double kSocTarget = 0.9;   // lpsolver.py:109
constexpr double kSocMax = 1.0;      // lpsolver.py:103
constexpr double kCountTol = 1e-9;
constexpr double kQpTol = 1e-11;     // KKT / feasibility tolerance of the utility QP
constexpr int kQpInnerMax = 60;      // Newton steps per launch
constexpr int kQpRoundMax = 400;     // working-set rounds per utility solve
constexpr int kDenseMaxN = 2048;     // zones above this size get no dense sensitivity block at all: tree input, tree-Newton path

struct Counters {
    int n_running;   // n_running and n_cls are reset together before every working-set round
    int n_cls[kQpClasses];
    int n_failed;
    int infeasible;
    int max_ws;
    unsigned long long newton_its;
    unsigned long long qp_flops;
    unsigned long long qp_cols;
    unsigned long long dbg[4 + 5 * kQpClasses];
    ResidualOut res;
    int round;       // working-set round of the current utility solve (device-side loop)
    int noconv;      // a utility solve hit kQpRoundMax rounds
    int iter;        // ADMM iterations done (device-side loop; selects the ping-pong side of the schedules)
    int pad_;
    unsigned long long rounds_total;   // working-set rounds since revs_admm_begin
};

struct ZoneGroups {  // static: which warp-kernel instantiations the zone sizes of this solver need
    int max_n = 0, warp_n = 0, n_small = 0, n_mid = 0, n_big = 0, mid_max = 0;
};

struct Tree {
    int n_nodes = 0;
    int* d_parent = nullptr;
    double* d_cumr = nullptr;
    int* d_res_node = nullptr;
    bool pooled = false;     // sub-range of the solver's tree pool (revs_set_feeder_trees)
};

template <class Tp>
cudaError_t dalloc(Tp** p, size_t n) {
    cudaError_t e = cudaMalloc((void**)p, (n ? n : 1) * sizeof(Tp));
    if (e == cudaSuccess) e = cudaMemset(*p, 0, (n ? n : 1) * sizeof(Tp));
    return e;
}

// One device array with one owner (move-only): freed when it is reallocated, replaced or destroyed.
template <class Tp>
struct DevArray {
    Tp* p = nullptr;
    DevArray& operator=(DevArray&& o) noexcept {
        std::swap(p, o.p);    // o frees the previous array
        return *this;
    }
    ~DevArray() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t n) {    // n elements, zeroed when it returns
        *this = DevArray();
        cudaError_t e = dalloc(&p, n);
        // dalloc zeroes on the legacy stream, which does not order with the non-blocking streams of the kernels
        return e == cudaSuccess ? cudaStreamSynchronize(cudaStreamLegacy) : e;
    }
    cudaError_t upload(const std::vector<Tp>& v) {    // alloc(v.size()) holding v
        cudaError_t e = alloc(v.size());
        if (e == cudaSuccess && !v.empty()) e = cudaMemcpy(p, v.data(), sizeof(Tp) * v.size(), cudaMemcpyHostToDevice);
        return e;
    }
    operator Tp*() const { return p; }
};

// The breadth-first zone arrays of the network tools (network_check.cu) and revs_network_check's arrays sized by the
// total node count: built by net_prepare from the trees, replaced as a whole when the trees change.
struct NetArrays {
    NetHost h;
    DevArray<NetZone> zones;
    DevArray<NetNode> nodes;
    DevArray<int> levels, res, lists, zone_cta;
    DevArray<NetCta> ctas;
    DevArray<NetPartial> part, sum;
    DevArray<double> zw, gstate;             // [zones][3] zone_worst; state of the zones above kNetSmemMax
    DevArray<double> cumr;                   // [total nodes] cumulative resistances in the zones' order
    DevArray<double> scale, volt, load;      // revs_network_check's scale, voltage and loading, on first use
    // revs_hosting_capacity's CTAs (two doubles of state per node and step: their own step grouping) and per-node
    // {W, N}, on its first call
    HcHost hc;
    bool hc_ready = false;
    DevArray<HcCta> hc_ctas;
    DevArray<int> hc_lists, hc_zone_cta;
    DevArray<double2> hc_wn;
    DevArray<double> hc_gstate;
    DevArray<unsigned long long> hc_part;    // [hosting CTAs][3]
};

enum NetTool { kNetHostCheck, kNetRepair, kNetCentral, kNetCertify, kNetHosting, kNetTools };

// State of the network tools (revs_network_check, revs_repair_schedule, revs_central_bracket, revs_certify_infeasible,
// revs_hosting_capacity).
// Everything but the zone arrays is allocated on a tool's first call by net_alloc and kept until revs_destroy.
struct NetTools {
    bool valid = false;                      // bf matches the trees
    bool ready[kNetTools] = {};              // net_alloc has run for the tool
    NetArrays bf;
    // [Hp][T] scratch, as many as the bracket uses: no call reads a word of it that the same call did not write
    DevArray<double> scratch[9];
    // the kept schedules, never scratch: REVS_NET_REPAIRED until the next ADMM run begins, REVS_NET_CENTRAL until the
    // homes, tariff or trees change
    DevArray<double> repaired, central;      // [Hp][T]
    bool repaired_valid = false, central_valid = false;
    // built once from the feeder sizes and T, which revs_create fixes
    DevArray<int> hzone;                     // [Hp] zone of every padded home row, -1: padding
    DevArray<int64_t> rep_wsoff;             // [zones] the repair kernel's state: shared memory (-1, at most rep_smem
    DevArray<char> rep_gws;                  // bytes) up to kRepairSmemMaxN residences, else at this offset of rep_gws
    size_t rep_smem = 0;
    // per-zone results and flags, read by no later call
    DevArray<int32_t> info;                  // [3][zones][3] the repair's zone_info; the bracket's two repairs and result
    DevArray<int> flag;                      // [1] the bracket's and the certificate's error flags
    DevArray<double> cen_sums, cen_bounds;   // [3][zones] cost1, cost2, C_max; [zones][2]
    DevArray<CenZone> cen_state;
    DevArray<int> crt_hpos;                  // [Hp]
    DevArray<int32_t> crt_cert;              // [zones][4]
    DevArray<unsigned long long> crt_key;    // [zones]
    DevArray<double> hc_cap, hc_uni;         // [Hp][T] home_cap (on first use); [zones][T] zone_uniform
    DevArray<int64_t> hc_counts;             // [zones][3]
};

struct TimedSpan { cudaEvent_t a, b; int cat; };

inline double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// Host-to-device uploads of the solvers that share one GPU take the PCIe link one at a time (parallel.PipelinedSolver
// runs one host thread per pipeline): the host-side preparation of every pipeline runs concurrently, and the pipeline
// whose inputs are complete starts computing while the next one is still uploading.
std::mutex& upload_mutex(int device) {
    static std::mutex mu[64];
    return mu[device & 63];
}

}  // namespace

struct revs_solver {
    int device = 0, nf = 0, T = 0, ncols = 0;
    int64_t H = 0, Hp = 0;
    std::vector<int64_t> off;            // compact home offsets [nf+1]
    std::vector<FeederDev> feeders;
    std::vector<char> sens_set;
    std::vector<Tree> trees;
    bool homes_set = false, tariff_set = false;

    FeederDev* d_feeders = nullptr;
    double* d_Rpool = nullptr;
    double* d_rn2 = nullptr;
    double* d_rmax = nullptr;
    int* d_cand = nullptr;
    double* d_stage = nullptr;                 // compact staging [H][T+1] for host transfers
    int64_t* d_hmap = nullptr;                 // compact home -> padded home
    void *d_Rbf = nullptr, *d_gbf = nullptr;   // BF16 copies for the screening contraction
    float* d_v32 = nullptr;
    ScreenProblem* d_sprob = nullptr;
    ContractTile* d_stiles = nullptr;
    int n_stiles = 0;
    ZoneGroups zg;
    // tuning / debug options, read ONCE (environment at revs_create, revs_set_option afterwards): nothing in the
    // solve path calls getenv
    int warp_m_max = 0, warp_m_max_big = 0;    // warm working sets above this size start in CTA class 1
    bool use_fast = true;                      // one-row register kernel for the small zones
    bool debug = false, debug_host = false;    // REVS_DEBUG / REVS_DEBUG_HOST: per-round / per-solve lines on stderr
    int trace_iter = -1, trace_round = -1;     // REVS_DEBUG_TRACE="<admm iteration>,<round>": per-column timeline of that round
    std::string trace_file = "revs_trace.bin"; // ... written here (REVS_DEBUG_TRACE_FILE), [ncols][12] int64
    bool use_graph = true;                     // revs_solve_admm: whole loop from one captured graph, loops decided on the device
    double host_sync_ms = 0.0, cat_ms[16] = {0};   // host time waiting in round syncs / span sums per category (debug_host)
    // captured ADMM loop (capture_loop): rebuilt when a parameter baked into it changes
    cudaGraph_t loop_graph = nullptr;
    cudaGraphExec_t loop_exec = nullptr;
    double gk_kappa = 0, gk_vset = 0, gk_vhigh = 0, gk_tol = 0;
    int gk_iter_max = 0, gk_flags = -1;
    double* d_respart = nullptr;               // per-CTA partial residual sums of dual_update_kernel
    double* d_dsum = nullptr;                  // [Hp] per-home sums of (P_sch[k+1] - P_sch[k])^2, home_solve_kernel -> dual_update_kernel
    // all-reduce of the residual sums over the GPUs of the box (revs_comm_*): peer-mapped mailboxes
    PeerSlot* d_mailbox = nullptr;             // [2][kMaxPeers] on this device, exported by IPC handle
    PeerSlot* peer_box[kMaxPeers] = {};        // mailboxes of all ranks as mapped into this process (peer_box[rank] == d_mailbox)
    int comm_world = 1, comm_rank = 0;
    unsigned long long comm_run = 0;           // run sequence, advanced by every revs_admm_begin on every rank alike
    unsigned long long* d_run_seq = nullptr;
    int* d_comm_timeout = nullptr;
    // large radial zones (tree_newton.cu): one CTA per column, products and active-set solves on the tree, no dense block
    int newton_min_n = 512;                    // zones given as TREES with more residences than this take that path (option "newton_min_n")
    std::vector<int64_t> roff_alloc;           // per feeder: its block in the R pool, -1 for zones above kDenseMaxN (tree input only)
    std::vector<char> is_newton;               // per feeder
    std::vector<NewtonZoneHost> nt_host;       // per feeder: breadth-first arrays (filled by revs_set_feeder_tree(s))
    std::vector<NewtonZone> nt_zones;
    NewtonZone* d_nt_zones = nullptr;
    int *d_nt_lvl = nullptr, *d_nt_parent = nullptr, *d_nt_home = nullptr, *d_nt_hnode = nullptr, *d_nt_wsi = nullptr;
    int2 *d_nt_child = nullptr, *d_nt_homes = nullptr;
    double *d_nt_rho = nullptr, *d_nt_ws = nullptr;
    double4* d_nt_ws4 = nullptr;
    double2* d_nt_ws2 = nullptr;
    int64_t nt_ws_stride = 0;
    int n_newton_cols = 0;
    size_t nt_sig = 0;
    // one feeder's reliability check row-partitioned over the GPUs of the box (revs_gather_* / revs_reliability_sharded)
    double* d_gather = nullptr;                // this rank's gather buffer: payload [gather_cap] + kGatherMaxPeers arrival flags
    int64_t gather_cap = 0;
    double* peer_gather[kGatherMaxPeers] = {}; // every rank's buffer as mapped into this process
    int gather_world = 1, gather_rank = 0;
    unsigned long long gather_seq = 0;         // advanced by every sharded call on every rank alike
    GatherDev* d_gather_dev = nullptr;
    unsigned* d_gather_ticket = nullptr;
    int* d_gather_timeout = nullptr;
    bool use_warp_kernel = true;               // class 0: one warp per small column (utility_qp_warp.cu)
    bool overlap_home = true;                  // home solve on its own (low priority) stream beside the utility kernels
    bool screen = true;                        // BF16 screening + exact recheck instead of the FP64 contraction in the loop
    int screen_impl = 0;                       // 0: mma.sync kernel, 1: tcgen05/TMEM/TMA kernel
    void *d_maps_a = nullptr, *d_map_b = nullptr;   // CUtensorMap per feeder block / for the bf16 schedule
    int* d_bcol0 = nullptr;
    bool tc5_ready = false;
    int *d_pool_parent = nullptr, *d_pool_res = nullptr;   // revs_set_feeder_trees
    double* d_pool_cumr = nullptr;
    int64_t* d_pool_off = nullptr;
    size_t pool_nodes = 0;
    NetTools net;                              // network check, repair, bracket, certificate and hosting capacity
    size_t Rpool_elems = 0;
    bool rn2_valid = false;
    // home-major [Hp][T]
    double *d_load = nullptr, *d_pest = nullptr, *d_psch[2] = {nullptr, nullptr}, *d_gamma = nullptr,
           *d_pev = nullptr, *d_soc = nullptr;
    uint8_t* d_has_ev = nullptr;
    double *d_rating = nullptr, *d_capacity = nullptr, *d_initial = nullptr, *d_indconst = nullptr;
    int *d_start = nullptr, *d_end = nullptr, *d_nmin = nullptr, *d_nmax = nullptr, *d_zero_i = nullptr;
    double* d_cost = nullptr;
    // time-major [T][Hp]
    double *d_zt = nullptr, *d_lamt = nullptr, *d_gt = nullptr, *d_vt = nullptr;
    int *d_wcount = nullptr, *d_widx = nullptr, *d_status = nullptr, *d_innerok = nullptr, *d_cls = nullptr;
    int *d_order = nullptr, *d_order_count = nullptr;
    int4* d_order4 = nullptr;
    Counters* d_cnt = nullptr;
    Counters* h_cnt = nullptr;           // pinned mirror
    void* h_homes = nullptr;             // pinned staging of the per-home vectors (revs_set_homes)
    size_t h_homes_bytes = 0;
    double* d_diff = nullptr;
    int diff_cap = 0;
    ContractProblem* d_cprob = nullptr;
    ContractTile* d_ctiles = nullptr;
    int n_ctiles = 0;
    cudaStream_t sU = nullptr, sH = nullptr;
    cudaStream_t sQ[kQpClasses] = {};          // the larger QP classes run beside class 0
    cudaEvent_t evV = nullptr, evQ[kQpClasses] = {};
    cudaEvent_t evHomeDone = nullptr, evDualDone = nullptr, evT0 = nullptr, evT1 = nullptr;
    std::vector<TimedSpan> spans;
    size_t span_used = 0;

    // run state
    double kappa = 5.0, vset = 1.0, vlow = 0.95, vhigh = 1.05, tol = 0.0;
    int iter_max = 0, k = 0, cur = 0;
    int warm_cls = kQpClasses - 1;   // largest QP class the stored multipliers can need
    int prio_lo = 0, prio_hi = 0;    // stream priority range of the device
    int ws_bound = kWMax;            // upper bound of every stored working-set size (decides which classes the first round launches)
    bool running = false;
    revs_stats stats{};
};

namespace {

int use_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(REVS_ERR_CUDA, "no CUDA device: %s (this library has no CPU fallback)",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(REVS_ERR_ARG, "device %d out of range (0..%d)", device, n - 1);
    CU(cudaSetDevice(device));
    cudaDeviceProp pr;
    CU(cudaGetDeviceProperties(&pr, device));
    if (pr.major < 10)
        return fail(REVS_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    pr.major, pr.minor);
    return REVS_OK;
}

TimedSpan* span_begin(revs_solver* s, int cat, cudaStream_t st) {
    if (s->span_used == s->spans.size()) {
        TimedSpan sp;
        cudaEventCreate(&sp.a);
        cudaEventCreate(&sp.b);
        sp.cat = cat;
        s->spans.push_back(sp);
    }
    TimedSpan* sp = &s->spans[s->span_used++];
    sp->cat = cat;
    cudaEventRecord(sp->a, st);
    return sp;
}
void span_end(TimedSpan* sp, cudaStream_t st) { cudaEventRecord(sp->b, st); }

void spans_collect(revs_solver* s) {   // after the streams are synchronised
    for (size_t i = 0; i < s->span_used; ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, s->spans[i].a, s->spans[i].b) != cudaSuccess) continue;
        s->cat_ms[s->spans[i].cat & 15] += ms;
        switch (s->spans[i].cat) {
            case 0: s->stats.gemm_ms += ms; break;
            case 5: s->stats.gemm_ms += ms; s->stats.gemm_full_ms += ms; break;
            case 1: s->stats.home_ms += ms; break;
            case 2: s->stats.dual_ms += ms; break;
            case 3: case 9: s->stats.qp_ms += ms; break;
            case 6: s->stats.qp_ms += ms; s->stats.qp_init_ms += ms; break;
            case 7: case 8: s->stats.qp_ms += ms; s->stats.qp_warp_ms += ms; break;
            case 4: s->stats.qp_ms += ms; s->stats.qp_big_ms += ms; break;
        }
    }
    s->span_used = 0;
}

void count_window(double rating, double cap, double init, int* nmin, int* nmax) {
    double step = rating / cap;
    int lo = (int)std::ceil((kSocTarget - init) / step - kCountTol);
    int hi = (int)std::floor((kSocMax - init) / step + kCountTol);
    *nmin = lo < 0 ? 0 : lo;
    *nmax = hi;
}

// copy a compact host array [H][w] into the padded device layout [Hp][w] (and back): one
// transfer through a device staging buffer plus a scatter / gather kernel, independent of
// the number of feeders
int h2d_homes(revs_solver* s, double* dst, const double* src, int w) {
    if (s->H == 0) return REVS_OK;
    CU(cudaMemcpyAsync(s->d_stage, src, (size_t)s->H * w * sizeof(double), cudaMemcpyHostToDevice, s->sU));
    CU(launch_pack_rows(s->d_stage, dst, s->d_hmap, s->H, w, 1, s->sU));
    return REVS_OK;
}
int d2h_homes(const revs_solver* s, double* dst, const double* src, int w) {
    if (s->H == 0) return REVS_OK;
    CU(launch_pack_rows(src, s->d_stage, s->d_hmap, s->H, w, 0, s->sU));
    CU(cudaMemcpyAsync(dst, s->d_stage, (size_t)s->H * w * sizeof(double), cudaMemcpyDeviceToHost, s->sU));
    return REVS_OK;
}

// A schedule on the device (P, p_ev: [Hp][T]) to the caller in the compact home order: hour_mask [H][mask_words]
// charging bits and P_out [H][T], each when given; *launches counts both kernels.
int schedule_d2h(const revs_solver* s, const double* P, const double* p_ev, double* P_out, uint64_t* hour_mask,
                 int mask_words, int64_t* launches) {
    if (hour_mask && s->H > 0) {
        unsigned long long* d_mask = reinterpret_cast<unsigned long long*>(s->d_stage);     // H (T + 1) doubles >= H W words
        CU(launch_hour_mask(p_ev, s->d_hmap, s->H, s->T, d_mask, s->sU));
        ++*launches;
        CU(cudaMemcpyAsync(hour_mask, d_mask, (size_t)s->H * mask_words * sizeof(uint64_t), cudaMemcpyDeviceToHost, s->sU));
    }
    if (P_out && s->H > 0) {
        int rc = d2h_homes(s, P_out, P, s->T);
        if (rc) return rc;
        ++*launches;
    }
    return REVS_OK;
}

int check_ready(const revs_solver* s) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    if (!s->homes_set) return fail(REVS_ERR_ARG, "revs_set_homes has not been called");
    if (!s->tariff_set) return fail(REVS_ERR_ARG, "revs_set_tariff has not been called");
    for (int f = 0; f < s->nf; ++f)
        if (!s->sens_set[f]) return fail(REVS_ERR_ARG, "feeder %d has no sensitivity block", f);
    return REVS_OK;
}

// Zone-size groups, contraction / screening tile tables and tensor maps over the zones that have a dense block
// (everything but the tree-Newton zones).  Called by revs_create and again when option "newton_min_n" moves zones.
int build_tables(revs_solver* s) {
    const int n_feeders = s->nf, T = s->T;
    const int64_t hp = s->Hp;
    s->zg = ZoneGroups();
    for (int f = 0; f < n_feeders; ++f) {
        const int n = s->feeders[f].n;
        if (s->is_newton[f]) continue;
        s->zg.max_n = std::max(s->zg.max_n, n);
        if (n > qp_warp_max_n()) continue;
        s->zg.warp_n = std::max(s->zg.warp_n, n);
        if (n <= 128) ++s->zg.n_small;
        else if (n <= 256) { ++s->zg.n_mid; s->zg.mid_max = std::max(s->zg.mid_max, n); }
        else ++s->zg.n_big;
    }
    if (s->zg.max_n > kScreenMaxN) s->screen = false;    // the error bound of the BF16 screening pass (kScreenUp) holds up to kScreenMaxN terms
    void* old[] = {s->d_sprob, s->d_stiles, s->d_maps_a, s->d_bcol0, s->d_cprob, s->d_ctiles};
    for (void* q : old) if (q) cudaFree(q);
    s->d_sprob = nullptr; s->d_stiles = nullptr; s->d_maps_a = nullptr; s->d_bcol0 = nullptr; s->d_cprob = nullptr; s->d_ctiles = nullptr;
    s->tc5_ready = false;
    if (s->loop_exec) { cudaGraphExecDestroy(s->loop_exec); s->loop_exec = nullptr; }

    // contraction table: V_t = R_f * G_t for every feeder, BM-row tiles
    std::vector<ContractProblem> probs(n_feeders);
    std::vector<ContractTile> tiles;
    const int bm = contract_tile_rows(T);
    for (int f = 0; f < n_feeders; ++f) {
        const FeederDev& fd = s->feeders[f];
        if (fd.roff < 0) { probs[f] = ContractProblem{}; continue; }
        probs[f] = ContractProblem{s->d_Rpool + fd.roff, fd.np, fd.np, fd.np, s->d_gt + fd.off, hp,
                                   s->d_vt + fd.off, hp, nullptr, s->d_status + (size_t)f * T};
        for (int r0 = 0; r0 < fd.np; r0 += bm) tiles.push_back(ContractTile{f, r0});
    }
    {   // screening table: same products in BF16 -> FP32
        std::vector<ScreenProblem> sp(n_feeders);
        std::vector<ContractTile> st;
        const int sbm = screen_tile_rows();
        for (int f = 0; f < n_feeders; ++f) {
            const FeederDev& fd = s->feeders[f];
            if (fd.roff < 0) { sp[f] = ScreenProblem{}; continue; }
            sp[f] = ScreenProblem{(const char*)s->d_Rbf + 2 * fd.roff, fd.np, fd.np, fd.np,
                                  (const char*)s->d_gbf + 2 * fd.off, hp, s->d_v32 + fd.off, hp,
                                  s->d_status + (size_t)f * T, s->d_cand + (size_t)f * T};
            for (int r0 = 0; r0 < fd.np; r0 += sbm) st.push_back(ContractTile{f, r0});
        }
        s->n_stiles = (int)st.size();
        CU(dalloc(&s->d_sprob, sp.size()));
        CU(cudaMemcpy(s->d_sprob, sp.data(), sp.size() * sizeof(ScreenProblem), cudaMemcpyHostToDevice));
        CU(dalloc(&s->d_stiles, st.size()));
        CU(cudaMemcpy(s->d_stiles, st.data(), st.size() * sizeof(ContractTile), cudaMemcpyHostToDevice));
        // tensor maps of the tcgen05 implementation (same 128-row tiling)
        if (T <= (int)screen_tc5_box_rows_b() && screen_tc5_tile_rows() == sbm) {
            const size_t mb = screen_tc5_map_bytes();
            std::vector<unsigned char> maps((size_t)(n_feeders + 1) * mb);
            std::vector<int> bcol(n_feeders);
            bool ok = true;
            for (int f = 0; f < n_feeders && ok; ++f) {
                const FeederDev& fd = s->feeders[f];
                bcol[f] = (int)fd.off;
                if (fd.roff < 0) continue;
                ok = screen_tc5_encode(maps.data() + (size_t)f * mb, (const char*)s->d_Rbf + 2 * fd.roff, fd.np, fd.np, fd.np,
                                       screen_tc5_box_rows_a()) == cudaSuccess;
            }
            ok = ok && screen_tc5_encode(maps.data() + (size_t)n_feeders * mb, s->d_gbf, T, hp, hp, screen_tc5_box_rows_b()) == cudaSuccess;
            if (ok) {
                CU(cudaMalloc(&s->d_maps_a, maps.size()));
                CU(cudaMemcpy(s->d_maps_a, maps.data(), maps.size(), cudaMemcpyHostToDevice));
                s->d_map_b = nullptr;   // last entry of the same allocation
                CU(dalloc(&s->d_bcol0, (size_t)n_feeders));
                CU(cudaMemcpy(s->d_bcol0, bcol.data(), sizeof(int) * n_feeders, cudaMemcpyHostToDevice));
                s->tc5_ready = true;
                s->screen_impl = 1;       // sm_100a-native kernel by default
                if (getenv("REVS_SCREEN_TC5")) s->screen_impl = atoi(getenv("REVS_SCREEN_TC5"));
            }
        }
    }
    s->n_ctiles = (int)tiles.size();
    CU(dalloc(&s->d_cprob, probs.size()));
    CU(cudaMemcpy(s->d_cprob, probs.data(), probs.size() * sizeof(ContractProblem), cudaMemcpyHostToDevice));
    CU(dalloc(&s->d_ctiles, tiles.size()));
    CU(cudaMemcpy(s->d_ctiles, tiles.data(), tiles.size() * sizeof(ContractTile), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(s->d_feeders, s->feeders.data(), sizeof(FeederDev) * n_feeders, cudaMemcpyHostToDevice));
    return REVS_OK;
}

// moves a zone between the dense path and the tree-Newton path (the caller rebuilds the tables)
int set_newton(revs_solver* s, int f, bool on) {
    if (!on && s->roff_alloc[f] < 0) return fail(REVS_ERR_ARG, "zone %d has no dense block", f);
    s->is_newton[f] = on ? 1 : 0;
    s->feeders[f].roff = on ? (int64_t)-1 : s->roff_alloc[f];
    s->rn2_valid = false;
    return REVS_OK;
}

// Static pools and work arrays of the tree-Newton zones whose trees have been given; column list = their hours.
int rebuild_newton(revs_solver* s) {
    std::vector<int> lvl, parent, hlist, hnode;
    std::vector<int2> child, homes;
    std::vector<double> rho;
    s->nt_zones.clear();
    int col0 = 0;
    int64_t ws = 0;
    for (int f = 0; f < s->nf; ++f) {
        if (!s->is_newton[f] || s->nt_host[f].parent.empty()) continue;
        const NewtonZoneHost& Z = s->nt_host[f];
        NewtonZone z{};
        z.feeder = f;
        z.nn = (int)Z.parent.size();
        z.nlev = (int)Z.lvl.size() - 1;
        z.n = (int)Z.hlist.size();
        z.wn = std::max(z.nn, z.n);
        z.col0 = col0;
        z.node_off = (int64_t)parent.size();
        z.home_off = (int64_t)hlist.size();
        z.lvl_off = (int64_t)lvl.size();
        z.ws_off = ws;
        z.scale = Z.scale;
        lvl.insert(lvl.end(), Z.lvl.begin(), Z.lvl.end());
        parent.insert(parent.end(), Z.parent.begin(), Z.parent.end());
        hlist.insert(hlist.end(), Z.hlist.begin(), Z.hlist.end());
        hnode.insert(hnode.end(), Z.hnode.begin(), Z.hnode.end());
        rho.insert(rho.end(), Z.rho.begin(), Z.rho.end());
        for (int i = 0; i < z.nn; ++i) { child.push_back(make_int2(Z.child0[i], Z.nchild[i])); homes.push_back(make_int2(Z.home0[i], Z.nhome[i])); }
        col0 += s->T;
        ws += (int64_t)z.wn * s->T;
        s->nt_zones.push_back(z);
    }
    {   // the same zones as last time (a caller re-uploading its feeders every schedule): nothing to do
        size_t sig = 1469598103934665603ull;
        auto mix = [&](const void* q, size_t bytes) {
            const unsigned char* b = (const unsigned char*)q;
            for (size_t i = 0; i < bytes; ++i) sig = (sig ^ b[i]) * 1099511628211ull;
        };
        for (const NewtonZone& z : s->nt_zones) mix(&z.feeder, sizeof(int));
        mix(lvl.data(), lvl.size() * sizeof(int));
        mix(parent.data(), parent.size() * sizeof(int));
        mix(hlist.data(), hlist.size() * sizeof(int));
        mix(homes.data(), homes.size() * sizeof(int2));
        mix(rho.data(), rho.size() * sizeof(double));
        if (sig == s->nt_sig && col0 == s->n_newton_cols && (col0 == 0 || s->d_nt_ws)) return REVS_OK;
        s->nt_sig = sig;
    }
    void* old[] = {s->d_nt_zones, s->d_nt_lvl, s->d_nt_parent, s->d_nt_home, s->d_nt_hnode, s->d_nt_wsi, s->d_nt_child, s->d_nt_homes, s->d_nt_rho, s->d_nt_ws, s->d_nt_ws4, s->d_nt_ws2};
    for (void* q : old) if (q) cudaFree(q);
    s->d_nt_zones = nullptr; s->d_nt_lvl = nullptr; s->d_nt_parent = nullptr; s->d_nt_home = nullptr; s->d_nt_wsi = nullptr;
    s->d_nt_child = nullptr; s->d_nt_homes = nullptr; s->d_nt_hnode = nullptr; s->d_nt_rho = nullptr; s->d_nt_ws = nullptr; s->d_nt_ws4 = nullptr; s->d_nt_ws2 = nullptr;
    s->n_newton_cols = col0;
    s->nt_ws_stride = ws;
    if (s->loop_exec) { cudaGraphExecDestroy(s->loop_exec); s->loop_exec = nullptr; }   // the captured loop bakes the pointers in
    if (col0 == 0) return REVS_OK;
    CU(dalloc(&s->d_nt_zones, s->nt_zones.size()));
    CU(cudaMemcpy(s->d_nt_zones, s->nt_zones.data(), sizeof(NewtonZone) * s->nt_zones.size(), cudaMemcpyHostToDevice));
    CU(dalloc(&s->d_nt_lvl, lvl.size()));
    CU(cudaMemcpy(s->d_nt_lvl, lvl.data(), sizeof(int) * lvl.size(), cudaMemcpyHostToDevice));
    CU(dalloc(&s->d_nt_parent, parent.size()));
    CU(cudaMemcpy(s->d_nt_parent, parent.data(), sizeof(int) * parent.size(), cudaMemcpyHostToDevice));
    CU(dalloc(&s->d_nt_home, hlist.size()));
    CU(cudaMemcpy(s->d_nt_home, hlist.data(), sizeof(int) * hlist.size(), cudaMemcpyHostToDevice));
    CU(dalloc(&s->d_nt_hnode, hnode.size()));
    CU(cudaMemcpy(s->d_nt_hnode, hnode.data(), sizeof(int) * hnode.size(), cudaMemcpyHostToDevice));
    CU(dalloc(&s->d_nt_homes, homes.size()));
    CU(cudaMemcpy(s->d_nt_homes, homes.data(), sizeof(int2) * homes.size(), cudaMemcpyHostToDevice));
    CU(dalloc(&s->d_nt_child, child.size()));
    CU(cudaMemcpy(s->d_nt_child, child.data(), sizeof(int2) * child.size(), cudaMemcpyHostToDevice));
    CU(dalloc(&s->d_nt_rho, rho.size()));
    CU(cudaMemcpy(s->d_nt_rho, rho.data(), sizeof(double) * rho.size(), cudaMemcpyHostToDevice));
    CU(dalloc(&s->d_nt_ws, (size_t)ws * kNewtonWsDoubles));
    CU(dalloc(&s->d_nt_ws4, (size_t)ws * kNewtonWs4));
    CU(dalloc(&s->d_nt_ws2, (size_t)ws * kNewtonWs2));
    CU(dalloc(&s->d_nt_wsi, (size_t)ws * kNewtonWsInts));
    return REVS_OK;
}

bool newton_active(const revs_solver* s) { return s->n_newton_cols > 0; }
int dense_cols(const revs_solver* s) { return s->ncols - s->n_newton_cols; }   // columns the dense kernels solve

int launch_newton_stage(revs_solver* s, bool timed) {
    if (!newton_active(s)) return REVS_OK;
    NewtonParams N{};
    N.zones = s->d_nt_zones; N.n_zones = (int)s->nt_zones.size();
    N.lvl = s->d_nt_lvl; N.parent = s->d_nt_parent; N.child = s->d_nt_child; N.homes = s->d_nt_homes; N.rho = s->d_nt_rho; N.hlist = s->d_nt_home; N.hnode = s->d_nt_hnode;
    N.ws = s->d_nt_ws; N.ws4 = s->d_nt_ws4; N.ws2 = s->d_nt_ws2; N.wsi = s->d_nt_wsi; N.ws_stride = s->nt_ws_stride;
    N.feeders = s->d_feeders; N.z_t = s->d_zt; N.lam_t = s->d_lamt; N.g_t = s->d_gt;
    N.status = s->d_status; N.inner_ok = s->d_innerok; N.wcount = s->d_wcount;
    N.noconv = &s->d_cnt->noconv; N.newton_its = &s->d_cnt->newton_its; N.cols = &s->d_cnt->qp_cols; N.flops = &s->d_cnt->qp_flops;
    N.max_ws = &s->d_cnt->max_ws;
    N.T = s->T; N.Hp = s->Hp;
    N.u = s->vhigh * s->vhigh - s->vset * s->vset;
    N.tol = kQpTol;
    int* d_dbg = nullptr;
    double* d_trace = nullptr;
    if (s->debug && timed) {
        CU(dalloc(&d_dbg, (size_t)2 * s->n_newton_cols)); N.dbg_col = d_dbg;
        CU(dalloc(&d_trace, (size_t)64 * s->n_newton_cols)); N.dbg_trace = d_trace;
    }
    double* d_dump = nullptr;
    size_t dump_n = 0;
    if (s->debug && timed && getenv("REVS_NEWTON_DUMP") &&
        sscanf(getenv("REVS_NEWTON_DUMP"), "%d,%d,%d", &N.dbg_dump_col, &N.dbg_dump_outer, &N.dbg_dump_guess) == 3) {     // (debug only)
        int zi = 0;
        while (zi + 1 < (int)s->nt_zones.size() && N.dbg_dump_col >= s->nt_zones[zi + 1].col0) ++zi;
        dump_n = (size_t)8 * s->nt_zones[zi].nn;
        CU(dalloc(&d_dump, dump_n));
        N.dbg_dump = d_dump;
    }
    TimedSpan* sp = timed ? span_begin(s, 9, s->sU) : nullptr;
    CU(launch_tree_newton(N, s->n_newton_cols, s->sU));
    if (sp) span_end(sp, s->sU);
    s->stats.kernel_launches++;
    if (d_dump) {
        std::vector<double> hd(dump_n);
        CU(cudaStreamSynchronize(s->sU));
        CU(cudaMemcpy(hd.data(), d_dump, dump_n * sizeof(double), cudaMemcpyDeviceToHost));
        cudaFree(d_dump);
        char name[128];
        snprintf(name, sizeof name, "newton_dump_admm%d.bin", s->k);
        if (FILE* fp = fopen(name, "wb")) { fwrite(hd.data(), sizeof(double), dump_n, fp); fclose(fp); }
    }
    if (d_dbg) {
        std::vector<int> h((size_t)2 * s->n_newton_cols);
        CU(cudaStreamSynchronize(s->sU));
        CU(cudaMemcpy(h.data(), d_dbg, h.size() * sizeof(int), cudaMemcpyDeviceToHost));
        cudaFree(d_dbg);
        long long sum_s = 0, sum_i = 0;
        int max_s = 0, max_i = 0, arg_s = 0;
        for (int c = 0; c < s->n_newton_cols; ++c) {
            sum_s += h[2 * c]; sum_i += h[2 * c + 1];
            if (h[2 * c] > max_s) { max_s = h[2 * c]; arg_s = c; }
            max_i = std::max(max_i, h[2 * c + 1]);
        }
        float ms = 0.f;
        if (sp) cudaEventElapsedTime(&ms, sp->a, sp->b);
        if (max_s > 60) {
            std::vector<double> tr(64);
            CU(cudaMemcpy(tr.data(), d_trace + (size_t)64 * arg_s, 64 * sizeof(double), cudaMemcpyDeviceToHost));
            for (int i = 0; i < 16 && i <= h[2 * arg_s + 1]; ++i)
                fprintf(stderr, "[revs]   column %d outer %d: kkt %.3e solves %g step %g active %g\n", arg_s, i, tr[4 * i], tr[4 * i + 1], tr[4 * i + 2], tr[4 * i + 3]);
        }
        cudaFree(d_trace);
        fprintf(stderr, "[revs] admm %d tree-Newton: %d columns, tree solves mean %.1f max %d (column %d), outer iterations mean %.1f max %d, %.3f ms\n", s->k,
                s->n_newton_cols, (double)sum_s / s->n_newton_cols, max_s, arg_s, (double)sum_i / s->n_newton_cols, max_i, ms);
    }
    return REVS_OK;
}

QpParams qp_params(revs_solver* s) {
    QpParams Q{};
    Q.feeders = s->d_feeders;
    Q.Rpool = s->d_Rpool;
    Q.rn2 = s->d_rn2;
    Q.rmax = s->d_rmax;
    Q.cand = s->screen ? s->d_cand : nullptr;
    Q.queue = s->d_order_count + kQpLists;
    Q.sweep = 0;
    Q.list0 = kQpClasses;
    Q.nlists = kQpBuckets;
    Q.list_extra = -1;
    Q.warp_m_max = s->warp_m_max;
    Q.warp_m_max_big = s->warp_m_max_big;
    Q.z_t = s->d_zt;
    Q.lam_t = s->d_lamt;
    Q.g_t = s->d_gt;
    Q.v_t = s->d_vt;
    Q.v32_t = s->screen ? s->d_v32 : nullptr;
    Q.gbf_t = s->screen ? s->d_gbf : nullptr;
    Q.wcount = s->d_wcount;
    Q.widx = s->d_widx;
    Q.status = s->d_status;
    Q.inner_ok = s->d_innerok;
    Q.n_running = &s->d_cnt->n_running;
    Q.newton_its = &s->d_cnt->newton_its;
    Q.max_ws = &s->d_cnt->max_ws;
    Q.flops = &s->d_cnt->qp_flops;
    Q.cols = &s->d_cnt->qp_cols;
    Q.n_failed = &s->d_cnt->n_failed;
    Q.cls = s->d_cls;
    Q.n_cls = s->d_cnt->n_cls;
    Q.order = s->d_order;
    Q.order4 = s->d_order4;
    Q.order_count = s->d_order_count;
    Q.ncols = s->ncols;
    Q.trace = nullptr;
    Q.dbg = s->debug ? s->d_cnt->dbg : nullptr;
    Q.T = s->T;
    Q.Hp = s->Hp;
    Q.u = s->vhigh * s->vhigh - s->vset * s->vset;
    Q.tol = kQpTol;
    Q.inner_max = kQpInnerMax;
    Q.init = 0;
    Q.round_ctr = &s->d_cnt->round;
    Q.cond_round = 0;
    Q.use_cond = 0;
    return Q;
}

int prepare_sensitivity(revs_solver* s) {
    if (s->rn2_valid) return REVS_OK;
    CU(launch_row_norms(s->d_feeders, s->nf, s->d_Rpool, s->d_rn2, s->d_rmax, s->sU));
    CU(launch_to_bf16(s->d_Rpool, s->d_Rbf, s->Rpool_elems, s->sU));
    s->rn2_valid = true;
    s->stats.kernel_launches += 2;
    return REVS_OK;
}

int launch_init(revs_solver* s, QpParams Q, bool in_loop, bool timed) {
    // Start of the solve: working sets from the stored multipliers, class by their size,
    // g = [z - R lam]_+ for the new target -- one warp per column.
    Q.init = in_loop ? 2 : 0;                      // 2: dual_update_kernel prepared g, multipliers sit on the stored rows
    Q.order = nullptr;
    TimedSpan* sp = timed ? span_begin(s, 6, s->sU) : nullptr;
    CU(launch_qp_init(Q, s->use_warp_kernel ? qp_warp_max_n() : 0, s->sU));
    if (sp) span_end(sp, s->sU);
    return REVS_OK;
}

// kernels one working-set round launches when every class runs (launch accounting of the captured loop)
int round_launches(const revs_solver* s) {
    const bool warp = s->use_warp_kernel && s->zg.warp_n > 0;
    int n = 2 + (kQpClasses - 1) + 1;              // screening / contraction, work lists, CTA classes, round end
    if (warp) n += (s->zg.n_big > 0) + (s->zg.n_mid > 0) + (s->zg.n_small > 0 ? 1 + (s->use_fast ? 1 : 0) : 0);
    return n;
}

// One working-set round, enqueued without waiting: screening pass, work lists, the QP classes side by side.
// mode 0: first round of a solve, 1: later rounds, -1: by the device round counter (captured loop).
// use / grid: which CTA classes can have work and how many columns (host-driven loop); nullptr = all, full grids.
// timed: CUDA-event spans around the kernels (not inside a stream capture: event nodes are not allowed in loop bodies).
struct GateCapture {   // captured loop: CTA classes 2 and 3 sit behind IF nodes decided on the device
    cudaGraphConditionalHandle h[kQpClasses];
    cudaGraph_t body[kQpClasses];
};

int enqueue_round(revs_solver* s, QpParams& Q, int mode, const bool* use, const int* grid, bool timed, GateCapture* gc = nullptr) {
    const double thr = (1.0 - kScreenMargin) * Q.u;
    TimedSpan* sp = timed ? span_begin(s, mode == 0 ? 5 : 0, s->sU) : nullptr;   // round 0: every column is running
    if (s->n_stiles == 0) {
        // no zone with a dense block: nothing to contract
    } else if (s->screen) {
        if (s->screen_impl == 1 && s->tc5_ready)
            CU(launch_screen_tc5(s->d_sprob, s->d_stiles, s->n_stiles, s->d_maps_a,
                                 (const char*)s->d_maps_a + (size_t)s->nf * screen_tc5_map_bytes(), s->d_bcol0, s->T, thr, s->sU));
        else
            CU(launch_screen(s->d_sprob, s->d_stiles, s->n_stiles, s->T, thr, s->sU));
    } else {
        CU(launch_contract(s->d_cprob, s->d_ctiles, s->n_ctiles, s->T, kOutTimeMajor, 0.0, s->sU));
    }
    if (sp) span_end(sp, s->sU);
    s->stats.kernel_launches++;
    if (mode == 0) s->stats.gemm_full_launches++;
    CU(cudaMemsetAsync(&s->d_cnt->n_running, 0, (1 + kQpClasses) * sizeof(int), s->sU));
    CU(launch_order_columns(Q, mode, s->d_order, s->d_order_count, s->sU));
    s->stats.kernel_launches++;
    if (gc) {
        // classes 2 and 3 need 73 / 210 KB of shared memory per CTA: even an empty launch of them would wait for (or
        // evict) the warp kernels' CTAs, so in the captured loop they run only when their work list is not empty
        ClassGateParams G{};
        G.order_count = s->d_order_count;
        for (int cl = 0; cl < kQpClasses; ++cl) G.cond[cl] = (unsigned long long)gc->h[cl];
        G.first_gated = 2;
        CU(launch_class_gate(G, s->sU));
    }
    // the larger classes go first, each on its own stream, so that their long CTAs
    // overlap with the many short columns of the small classes
    CU(cudaEventRecord(s->evV, s->sU));
    for (int cl = kQpClasses - 1; cl >= 1; --cl) {
        if (use && !use[cl]) continue;
        CU(cudaStreamWaitEvent(s->sQ[cl], s->evV, 0));
        if (gc && cl >= 2) {
            cudaStreamCaptureStatus st;
            cudaGraph_t g_cap = nullptr;
            const cudaGraphNode_t* deps = nullptr;
            size_t n_deps = 0;
            CU(cudaStreamGetCaptureInfo(s->sQ[cl], &st, nullptr, &g_cap, &deps, &n_deps));
            cudaGraphNodeParams np{};
            np.type = cudaGraphNodeTypeConditional;
            np.conditional.handle = gc->h[cl];
            np.conditional.type = cudaGraphCondTypeIf;
            np.conditional.size = 1;
            cudaGraphNode_t node;
            CU(cudaGraphAddNode(&node, g_cap, deps, n_deps, &np));
            gc->body[cl] = np.conditional.phGraph_out[0];
            CU(cudaStreamUpdateCaptureDependencies(s->sQ[cl], &node, 1, cudaStreamSetCaptureDependencies));
            CU(cudaEventRecord(s->evQ[cl], s->sQ[cl]));
            continue;
        }
        sp = timed ? span_begin(s, cl == 1 ? 3 : 4, s->sQ[cl]) : nullptr;
        CU(launch_utility_qp(Q, grid ? grid[cl] : s->ncols, cl, s->sQ[cl]));
        if (sp) span_end(sp, s->sQ[cl]);
        CU(cudaEventRecord(s->evQ[cl], s->sQ[cl]));
        s->stats.kernel_launches++;
    }
    if ((!use || use[0]) && s->use_warp_kernel && s->zg.warp_n > 0) {
        // one persistent warp-per-column kernel per zone-size group, one after the other on the utility stream
        // (sharing the SMs between two QP kernels slowed both down whenever it was measured): the groups of
        // long columns first, the many short columns of the small zones fill the tail
        s->stats.qp_warp_rounds++;
        const int full = qp_warp_ctas_per_sm();
        if (s->zg.n_big > 0) {                                    // zones of 257..320 residences: lists 13..16
            Q.list0 = kListBig;
            Q.nlists = kQpBuckets;
            Q.list_extra = -1;
            sp = timed ? span_begin(s, 7, s->sU) : nullptr;
            CU(launch_utility_qp_warp(Q, 10, full, s->sU));
            if (sp) span_end(sp, s->sU);
            s->stats.kernel_launches++;
        }
        if (s->zg.n_mid > 0) {                                    // zones of 129..256 residences: lists 8..11
            Q.list0 = kQpClasses + kQpBuckets;
            Q.nlists = kQpBuckets;
            Q.list_extra = -1;
            sp = timed ? span_begin(s, 7, s->sU) : nullptr;
            CU(launch_utility_qp_warp(Q, s->zg.mid_max <= 192 ? 6 : 8, full, s->sU));
            if (sp) span_end(sp, s->sU);
            s->stats.kernel_launches++;
        }
        if (s->zg.n_small > 0) {
            // small zones: the one-row kernel first (short columns, twice the occupancy), then the general
            // kernel for the columns with two or more stored rows (hardest first) and what the first passed on
            sp = timed ? span_begin(s, 8, s->sU) : nullptr;
            if (s->use_fast) {
                CU(launch_utility_qp_fast(Q, s->sU));
                s->stats.kernel_launches++;
            }
            Q.list0 = kQpClasses;
            Q.nlists = s->use_fast ? 2 : kQpBuckets;
            Q.list_extra = s->use_fast ? kListLeftover : -1;
            CU(launch_utility_qp_warp(Q, 4, full, s->sU));
            Q.list_extra = -1;
            s->stats.kernel_launches++;
            if (sp) span_end(sp, s->sU);
        }
    }
    for (int cl = 1; cl < kQpClasses; ++cl)
        if (!use || use[cl]) CU(cudaStreamWaitEvent(s->sU, s->evQ[cl], 0));
    s->stats.gemm_launches++;
    s->stats.qp_outer_iterations++;
    return REVS_OK;
}

int check_device_flags(revs_solver* s) {
    if (s->h_cnt->infeasible)
        return fail(REVS_ERR_INFEASIBLE, "a home charging sub-problem is infeasible (SOC window vs plug-in window)");
    if (s->h_cnt->n_failed)
        return fail(REVS_ERR_NOCONV,
                    "utility QP: %d (feeder,hour) columns need more than %d simultaneously active "
                    "voltage rows", s->h_cnt->n_failed, kWMax);
    if (s->h_cnt->noconv)
        return fail(REVS_ERR_NOCONV, "utility QP: %d columns still running after %d working-set rounds (or a tree-Newton column "
                    "that did not reach the tolerance)", s->h_cnt->n_running, kQpRoundMax);
    return REVS_OK;
}

// One utility solve, driven from the host (one pinned counter block read back per working-set round):
// project z_t onto the voltage polytope of every (feeder,hour) column.  Used by revs_utility_step,
// revs_admm_step and the profiling mode of revs_solve_admm; the default revs_solve_admm runs the same
// kernels from a captured graph whose loops are decided on the device (capture_loop below).
int utility_solve(revs_solver* s, bool in_loop = false) {
    int rc = prepare_sensitivity(s);
    if (rc) return rc;
    QpParams Q = qp_params(s);
    if ((rc = launch_init(s, Q, in_loop, true))) return rc;
    s->stats.kernel_launches++;
    if (newton_active(s)) {
        if ((rc = launch_newton_stage(s, true))) return rc;
        if (dense_cols(s) == 0) {
            CU(cudaMemcpyAsync(s->h_cnt, s->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, s->sU));
            CU(cudaStreamSynchronize(s->sU));
            return check_device_flags(s);
        }
    }
    bool use[kQpClasses];
    // first round: qp_init_kernel assigns classes on the device by the size of the stored working
    // sets; the largest working set any column has had in this solve (read back at every round
    // sync) bounds them, so larger classes need no launch
    for (int cl = 0; cl < kQpClasses; ++cl) use[cl] = cl <= 1 || qp_class_cap(cl - 1) < s->ws_bound;
    int top_cls = 0;
    int grid[kQpClasses];
    for (int cl = 0; cl < kQpClasses; ++cl) grid[cl] = s->ncols;
    for (int round = 0;; ++round) {
        if (round >= kQpRoundMax)
            return fail(REVS_ERR_NOCONV, "utility QP: %d columns still running after %d working-set rounds",
                        s->h_cnt->n_running, round);
        long long* d_trace = nullptr;
        if (in_loop && s->k == s->trace_iter && round == s->trace_round) {
            CU(cudaMalloc(&d_trace, sizeof(long long) * 12 * s->ncols));
            CU(cudaMemsetAsync(d_trace, 0, sizeof(long long) * 12 * s->ncols, s->sU));
            Q.trace = d_trace;
        }
        if ((rc = enqueue_round(s, Q, round == 0 ? 0 : 1, use, grid, true))) return rc;
        if (d_trace) {
            std::vector<long long> hb((size_t)12 * s->ncols);
            CU(cudaStreamSynchronize(s->sU));
            CU(cudaMemcpy(hb.data(), d_trace, hb.size() * sizeof(long long), cudaMemcpyDeviceToHost));
            if (FILE* fp = fopen(s->trace_file.c_str(), "wb")) {
                fwrite(hb.data(), sizeof(long long), hb.size(), fp);
                fclose(fp);
            }
            cudaFree(d_trace);
            Q.trace = nullptr;
        }
        CU(cudaMemcpyAsync(s->h_cnt, s->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, s->sU));
        {
            const double t0 = now_ms();
            CU(cudaStreamSynchronize(s->sU));
            s->host_sync_ms += now_ms() - t0;
        }
        if ((rc = check_device_flags(s))) return rc;
        if (s->debug)
            fprintf(stderr, "[revs] admm %d round %d: running %d by class %d/%d/%d/%d pieces_total %llu max_ws %d | phi evals %llu "
                    "pdas guesses %llu max pieces/launch %llu fallbacks %llu\n",
                    s->k, round, s->h_cnt->n_running, s->h_cnt->n_cls[0], s->h_cnt->n_cls[1], s->h_cnt->n_cls[2], s->h_cnt->n_cls[3],
                    s->h_cnt->newton_its, s->h_cnt->max_ws, s->h_cnt->dbg[0], s->h_cnt->dbg[1], s->h_cnt->dbg[2],
                    s->h_cnt->dbg[3]);
        s->ws_bound = std::max(s->ws_bound, s->h_cnt->max_ws);
        if (s->h_cnt->n_running == 0) break;
        for (int cl = 0; cl < kQpClasses; ++cl) {
            // n_cls: columns of the class that are still running (or were handed to it)
            grid[cl] = s->h_cnt->n_cls[cl] < s->ncols ? s->h_cnt->n_cls[cl] : s->ncols;
            use[cl] = s->h_cnt->n_cls[cl] > 0;
            if (use[cl]) top_cls = cl;
        }
    }
    s->warm_cls = top_cls;
    if (s->debug && s->k == s->iter_max - 1)
        for (int cl = 0; cl < kQpClasses; ++cl) {
            const unsigned long long* p = s->h_cnt->dbg + 4 + 5 * cl;
            fprintf(stderr, "[revs] class %d phase Mcycles: grad+kkt %.1f hessian %.1f pdas %.1f search %.1f final-eval %.1f\n", cl,
                    p[0] * 1e-6, p[1] * 1e-6, p[2] * 1e-6, p[3] * 1e-6, p[4] * 1e-6);
        }
    return REVS_OK;
}

HomeParams home_params(revs_solver* s, int individual) {
    HomeParams P;
    P.load = s->d_load;
    P.p_est = s->d_pest;
    P.p_sch = s->d_psch[s->cur];
    P.iter = nullptr;
    P.gamma = s->d_gamma;
    P.cost = s->d_cost;
    P.has_ev = s->d_has_ev;
    P.rating = s->d_rating;
    P.start = s->d_start;
    P.end = s->d_end;
    P.n_min = individual ? s->d_zero_i : s->d_nmin;
    P.n_max = s->d_nmax;
    P.p_sch_new = s->d_psch[s->cur ^ 1];
    P.p_ev = s->d_pev;
    P.infeasible = &s->d_cnt->infeasible;
    P.Hp = (int)s->Hp;
    P.T = s->T;
    P.kappa = s->kappa;
    P.individual = individual;
    P.ind_const = s->d_indconst;
    P.dsum = nullptr;              // set by the ADMM loop (revs_admm_step / capture_loop)
    P.first = 0;
    return P;
}

void free_all(revs_solver* s) {
    cudaSetDevice(s->device);
    void* ptrs[] = {s->d_feeders, s->d_Rpool, s->d_rn2, s->d_rmax, s->d_cand, s->d_stage, s->d_hmap, s->d_Rbf, s->d_gbf, s->d_v32, s->d_sprob, s->d_stiles, s->d_maps_a, s->d_map_b, s->d_bcol0, s->d_pool_parent, s->d_pool_res, s->d_pool_cumr, s->d_pool_off, s->d_load, s->d_pest, s->d_psch[0], s->d_psch[1], s->d_gamma,
                    s->d_pev, s->d_soc, s->d_has_ev, s->d_rating, s->d_capacity, s->d_initial, s->d_indconst,
                    s->d_start, s->d_end, s->d_nmin, s->d_nmax, s->d_zero_i, s->d_cost, s->d_zt, s->d_lamt,
                    s->d_gt, s->d_vt, s->d_wcount, s->d_widx, s->d_status, s->d_innerok, s->d_cls, s->d_order, s->d_order4, s->d_order_count, s->d_cnt, s->d_diff,
                    s->d_cprob, s->d_ctiles, s->d_respart, s->d_dsum,
                    s->d_nt_zones, s->d_nt_lvl, s->d_nt_parent, s->d_nt_home, s->d_nt_hnode, s->d_nt_wsi, s->d_nt_child, s->d_nt_homes, s->d_nt_rho,
                    s->d_nt_ws, s->d_nt_ws4, s->d_nt_ws2};
    for (int r = 0; r < kMaxPeers; ++r)
        if (s->peer_box[r] && s->peer_box[r] != s->d_mailbox) cudaIpcCloseMemHandle(s->peer_box[r]);
    for (int r = 0; r < kGatherMaxPeers; ++r)
        if (s->peer_gather[r] && s->peer_gather[r] != s->d_gather) cudaIpcCloseMemHandle(s->peer_gather[r]);
    if (s->d_gather) cudaFree(s->d_gather);
    if (s->d_gather_dev) cudaFree(s->d_gather_dev);
    if (s->d_gather_ticket) cudaFree(s->d_gather_ticket);
    if (s->d_gather_timeout) cudaFree(s->d_gather_timeout);
    if (s->d_mailbox) cudaFree(s->d_mailbox);
    if (s->d_run_seq) cudaFree(s->d_run_seq);
    if (s->d_comm_timeout) cudaFree(s->d_comm_timeout);
    if (s->loop_exec) cudaGraphExecDestroy(s->loop_exec);
    if (s->loop_graph) cudaGraphDestroy(s->loop_graph);
    for (void* p : ptrs)
        if (p) cudaFree(p);
    for (auto& t : s->trees) {
        if (t.pooled) continue;
        if (t.d_parent) cudaFree(t.d_parent);
        if (t.d_cumr) cudaFree(t.d_cumr);
        if (t.d_res_node) cudaFree(t.d_res_node);
    }
    if (s->h_cnt) cudaFreeHost(s->h_cnt);
    if (s->h_homes) cudaFreeHost(s->h_homes);
    for (auto& sp : s->spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    if (s->evHomeDone) cudaEventDestroy(s->evHomeDone);
    if (s->evDualDone) cudaEventDestroy(s->evDualDone);
    if (s->evT0) cudaEventDestroy(s->evT0);
    if (s->evT1) cudaEventDestroy(s->evT1);
    if (s->evV) cudaEventDestroy(s->evV);
    for (int cl = 0; cl < kQpClasses; ++cl) {
        if (s->evQ[cl]) cudaEventDestroy(s->evQ[cl]);
        if (s->sQ[cl]) cudaStreamDestroy(s->sQ[cl]);
    }
    if (s->sU) cudaStreamDestroy(s->sU);
    if (s->sH) cudaStreamDestroy(s->sH);
}

}  // namespace

extern "C" {

const char* revs_last_error(void) { return g_err.c_str(); }
int revs_version(void) { return 100; }

int revs_device_count(int* count) {
    if (!count) return fail(REVS_ERR_ARG, "null pointer");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *count = 0; return fail(REVS_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
    *count = n;
    return REVS_OK;
}

int revs_create(revs_solver** out, int device, int n_feeders, const int64_t* feeder_off, int T) {
    if (!out || !feeder_off || n_feeders <= 0 || T <= 0) return fail(REVS_ERR_ARG, "bad arguments");
    if (T > 256) return fail(REVS_ERR_ARG, "horizon T=%d exceeds the supported 256 steps", T);
    if (feeder_off[0] != 0) return fail(REVS_ERR_ARG, "feeder_off[0] must be 0");
    for (int f = 0; f < n_feeders; ++f)
        if (feeder_off[f + 1] < feeder_off[f]) return fail(REVS_ERR_ARG, "feeder_off must be non-decreasing");
    int rc = use_device(device);
    if (rc) return rc;

    revs_solver* s = new revs_solver();
    s->device = device;
    s->nf = n_feeders;
    s->T = T;
    s->ncols = n_feeders * T;
    s->off.assign(feeder_off, feeder_off + n_feeders + 1);
    s->H = feeder_off[n_feeders];
    s->feeders.resize(n_feeders);
    s->sens_set.assign(n_feeders, 0);
    s->trees.resize(n_feeders);
    s->is_newton.assign(n_feeders, 0);
    s->nt_host.resize(n_feeders);
    s->roff_alloc.assign(n_feeders, -1);
    if (const char* e = getenv("REVS_NEWTON_MIN_N")) s->newton_min_n = atoi(e);
    int64_t hp = 0, rp = 0;
    for (int f = 0; f < n_feeders; ++f) {
        int64_t n = feeder_off[f + 1] - feeder_off[f];
        int64_t np = (n + kPad - 1) / kPad * kPad;
        if (np == 0) np = kPad;
        // zones above kDenseMaxN residences run on the tree only (tree_newton.cu): no n^2 block for them
        s->is_newton[f] = n > kDenseMaxN;
        s->roff_alloc[f] = s->is_newton[f] ? (int64_t)-1 : rp;
        s->feeders[f] = FeederDev{(int)n, (int)np, hp, s->roff_alloc[f]};
        hp += np;
        if (!s->is_newton[f]) rp += np * np;
    }
    s->Hp = hp;
    const size_t HT = (size_t)hp * T;

#define TRY(x)                                                                                     \
    do {                                                                                           \
        cudaError_t e_ = (x);                                                                      \
        if (e_ != cudaSuccess) {                                                                   \
            free_all(s);                                                                           \
            delete s;                                                                              \
            return fail(REVS_ERR_CUDA, "%s failed: %s", #x, cudaGetErrorString(e_));               \
        }                                                                                          \
    } while (0)
    // the operator side is the critical path of an iteration; the home solve only has to be done
    // by the dual update, so its CTAs yield the SMs to the utility kernels
    int prio_lo = 0, prio_hi = 0;
    TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    s->prio_lo = prio_lo;
    s->prio_hi = prio_hi;
    TRY(cudaStreamCreateWithPriority(&s->sU, cudaStreamNonBlocking, prio_hi));
    TRY(cudaStreamCreateWithPriority(&s->sH, cudaStreamNonBlocking, prio_lo));
    TRY(cudaEventCreateWithFlags(&s->evV, cudaEventDisableTiming));
    for (int cl = 0; cl < kQpClasses; ++cl) {
        TRY(cudaStreamCreateWithPriority(&s->sQ[cl], cudaStreamNonBlocking, prio_hi));
        TRY(cudaEventCreateWithFlags(&s->evQ[cl], cudaEventDisableTiming));
    }
    TRY(cudaEventCreateWithFlags(&s->evHomeDone, cudaEventDisableTiming));
    TRY(cudaEventCreateWithFlags(&s->evDualDone, cudaEventDisableTiming));
    TRY(cudaEventCreate(&s->evT0));
    TRY(cudaEventCreate(&s->evT1));
    TRY(dalloc(&s->d_feeders, (size_t)n_feeders));
    TRY(cudaMemcpy(s->d_feeders, s->feeders.data(), sizeof(FeederDev) * n_feeders, cudaMemcpyHostToDevice));
    TRY(dalloc(&s->d_Rpool, (size_t)rp));
    TRY(dalloc(&s->d_rn2, (size_t)hp));
    TRY(dalloc(&s->d_rmax, (size_t)hp));
    TRY(dalloc(&s->d_cand, (size_t)s->ncols));
    TRY(dalloc(&s->d_stage, (size_t)s->H * (T + 1)));
    {
        std::vector<int64_t> hmap((size_t)s->H);
        for (int f = 0; f < n_feeders; ++f)
            for (int64_t i = feeder_off[f]; i < feeder_off[f + 1]; ++i) hmap[i] = s->feeders[f].off + (i - feeder_off[f]);
        TRY(dalloc(&s->d_hmap, hmap.size()));
        TRY(cudaMemcpy(s->d_hmap, hmap.data(), hmap.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
    }
    s->Rpool_elems = (size_t)rp;
    TRY(cudaMalloc(&s->d_Rbf, (size_t)(rp ? rp : 1) * 2));
    TRY(cudaMemset(s->d_Rbf, 0, (size_t)(rp ? rp : 1) * 2));
    TRY(cudaMalloc(&s->d_gbf, HT * 2));
    TRY(cudaMemset(s->d_gbf, 0, HT * 2));
    TRY(dalloc(&s->d_v32, HT));
    if (getenv("REVS_EXACT_GEMM")) s->screen = false;          // (create time only)
    TRY(dalloc(&s->d_load, HT));
    TRY(dalloc(&s->d_pest, HT));
    TRY(dalloc(&s->d_psch[0], HT));
    TRY(dalloc(&s->d_psch[1], HT));
    TRY(dalloc(&s->d_gamma, HT));
    TRY(dalloc(&s->d_pev, HT));
    TRY(dalloc(&s->d_soc, (size_t)hp * (T + 1)));
    TRY(dalloc(&s->d_has_ev, (size_t)hp));
    TRY(dalloc(&s->d_rating, (size_t)hp));
    TRY(dalloc(&s->d_capacity, (size_t)hp));
    TRY(dalloc(&s->d_initial, (size_t)hp));
    TRY(dalloc(&s->d_indconst, (size_t)hp));
    TRY(dalloc(&s->d_start, (size_t)hp));
    TRY(dalloc(&s->d_end, (size_t)hp));
    TRY(dalloc(&s->d_nmin, (size_t)hp));
    TRY(dalloc(&s->d_nmax, (size_t)hp));
    TRY(dalloc(&s->d_zero_i, (size_t)hp));
    TRY(dalloc(&s->d_cost, (size_t)T));
    TRY(dalloc(&s->d_zt, HT));
    TRY(dalloc(&s->d_lamt, HT));
    TRY(dalloc(&s->d_gt, HT));
    TRY(dalloc(&s->d_vt, HT));
    TRY(dalloc(&s->d_wcount, (size_t)s->ncols));
    TRY(dalloc(&s->d_widx, (size_t)s->ncols * kWMax));
    TRY(dalloc(&s->d_status, (size_t)s->ncols));
    TRY(dalloc(&s->d_innerok, (size_t)s->ncols));
    TRY(dalloc(&s->d_cls, (size_t)s->ncols));
    TRY(dalloc(&s->d_order, (size_t)s->ncols * kQpClasses));
    TRY(dalloc(&s->d_order4, (size_t)s->ncols * (kQpLists - kQpClasses)));
    if (hp >= (int64_t)1 << 31 || (rp >> 4) >= (int64_t)1 << 31) s->use_warp_kernel = false;   // 32-bit work-list entries
    TRY(dalloc(&s->d_order_count, (size_t)2 * kQpLists));
    TRY(dalloc(&s->d_cnt, (size_t)1));
    TRY(dalloc(&s->d_respart, (size_t)2 * ((hp + 31) / 32)));
    TRY(dalloc(&s->d_dsum, (size_t)hp));
    // options from the environment, read here and nowhere else
    {
        const char* e;
        s->warp_m_max = (e = getenv("REVS_WARP_M_MAX")) ? atoi(e) : qp_warp_m_max_default();
        // zones above 128 residences: the same threshold (round 1 sent stored sets above 5 rows to the first CTA class, which
        // cost 8.5 of 21 ms per schedule on zones of 150..300 residences; measured, profiles/README_r02.md)
        s->warp_m_max_big = (e = getenv("REVS_WARP_M_MAX_BIG")) ? atoi(e) : s->warp_m_max;
        s->use_fast = !((e = getenv("REVS_NO_FAST")) && atoi(e));
        s->debug = getenv("REVS_DEBUG") != nullptr;
        s->debug_host = getenv("REVS_DEBUG_HOST") != nullptr;
        if ((e = getenv("REVS_NO_GRAPH")) && atoi(e)) s->use_graph = false;
        if ((e = getenv("REVS_DEBUG_TRACE")) && sscanf(e, "%d,%d", &s->trace_iter, &s->trace_round) == 2) s->use_graph = false;
        if ((e = getenv("REVS_DEBUG_TRACE_FILE"))) s->trace_file = e;
        if (s->debug) s->use_graph = false;      // the per-round lines need the host-driven loop
    }
    TRY(cudaHostAlloc((void**)&s->h_cnt, sizeof(Counters), cudaHostAllocDefault));
    memset(s->h_cnt, 0, sizeof(Counters));

    {
        int rc2 = build_tables(s);
        if (rc2) { free_all(s); delete s; return rc2; }
    }
#undef TRY
    *out = s;
    return REVS_OK;
}

int revs_destroy(revs_solver* s) {
    if (!s) return REVS_OK;
    free_all(s);
    delete s;
    return REVS_OK;
}

int revs_set_sensitivity(revs_solver* s, int feeder, const double* R_res) {
    if (!s || !R_res || feeder < 0 || feeder >= s->nf) return fail(REVS_ERR_ARG, "bad arguments");
    CU(cudaSetDevice(s->device));
    const FeederDev& fd = s->feeders[feeder];
    if (s->roff_alloc[feeder] < 0)
        return fail(REVS_ERR_ARG, "feeder %d has %d residences (> %d): it runs on its tree, give it with "
                    "revs_set_feeder_tree(s) instead of a dense block", feeder, fd.n, kDenseMaxN);
    if (s->is_newton[feeder]) {          // a dense block replaces the tree: back to the dense kernels
        int rc = set_newton(s, feeder, false);
        if (rc) return rc;
        s->nt_host[feeder] = NewtonZoneHost();
        if ((rc = build_tables(s)) || (rc = rebuild_newton(s))) return rc;
    }
    for (int64_t i = 0; i < (int64_t)fd.n * fd.n; ++i)
        if (!(R_res[i] >= 0.0)) return fail(REVS_ERR_ARG, "sensitivity block of feeder %d has a negative or NaN entry", feeder);
    if (fd.n)
        CU(cudaMemcpy2D(s->d_Rpool + fd.roff, (size_t)fd.np * sizeof(double), R_res, (size_t)fd.n * sizeof(double),
                        (size_t)fd.n * sizeof(double), fd.n, cudaMemcpyHostToDevice));
    s->sens_set[feeder] = 1;
    s->rn2_valid = false;
    return REVS_OK;
}

int revs_set_feeder_tree(revs_solver* s, int feeder, int n_nodes, const int32_t* parent, const double* r,
                         const int32_t* res_node) {
    if (!s || !parent || !r || !res_node || feeder < 0 || feeder >= s->nf || n_nodes <= 0)
        return fail(REVS_ERR_ARG, "bad arguments");
    CU(cudaSetDevice(s->device));
    const FeederDev& fd = s->feeders[feeder];
    std::vector<double> cumr(n_nodes);
    for (int i = 0; i < n_nodes; ++i) {
        if (parent[i] >= i || parent[i] < -1) return fail(REVS_ERR_ARG, "nodes must be topologically ordered (parent[i] < i)");
        if (!(r[i] >= 0.0)) return fail(REVS_ERR_ARG, "negative or NaN resistance at node %d", i);
        cumr[i] = (parent[i] < 0 ? 0.0 : cumr[parent[i]]) + r[i];
    }
    for (int j = 0; j < fd.n; ++j)
        if (res_node[j] < 0 || res_node[j] >= n_nodes) return fail(REVS_ERR_ARG, "res_node[%d] out of range", j);
    Tree& t = s->trees[feeder];
    if (t.d_parent && !t.pooled) { cudaFree(t.d_parent); cudaFree(t.d_cumr); cudaFree(t.d_res_node); }
    t = Tree();
    s->net.valid = false;
    s->net.central_valid = false;
    t.n_nodes = n_nodes;
    CU(dalloc(&t.d_parent, (size_t)n_nodes));
    CU(dalloc(&t.d_cumr, (size_t)n_nodes));
    CU(dalloc(&t.d_res_node, (size_t)fd.np));
    CU(cudaMemcpy(t.d_parent, parent, sizeof(int) * n_nodes, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(t.d_cumr, cumr.data(), sizeof(double) * n_nodes, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(t.d_res_node, res_node, sizeof(int) * fd.n, cudaMemcpyHostToDevice));
    {
        const bool want = fd.n > s->newton_min_n || s->roff_alloc[feeder] < 0;
        if (want != (bool)s->is_newton[feeder]) {
            int rc = set_newton(s, feeder, want);
            if (rc || (rc = build_tables(s))) return rc;
        }
    }
    if (s->is_newton[feeder]) {
        newton_build_zone(n_nodes, parent, r, fd.n, res_node, s->nt_host[feeder]);
        s->sens_set[feeder] = 1;
        return rebuild_newton(s);
    }
    CU(launch_sens_voltage(t.d_parent, t.d_cumr, nullptr, t.d_res_node, fd.n, fd.n, s->d_Rpool + fd.roff, fd.np, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    s->sens_set[feeder] = 1;
    s->rn2_valid = false;
    return REVS_OK;
}

int revs_set_feeder_trees(revs_solver* s, const int64_t* node_off, const int32_t* parent, const double* r,
                          const int32_t* res_node) {
    if (!s || !node_off || !parent || !r || !res_node) return fail(REVS_ERR_ARG, "bad arguments");
    const double th0 = now_ms();
    CU(cudaSetDevice(s->device));
    if (node_off[0] != 0) return fail(REVS_ERR_ARG, "node_off[0] must be 0");
    const int64_t total = node_off[s->nf];
    std::vector<double> cumr((size_t)total);
    std::vector<int> res_p((size_t)s->Hp, 0);
    for (int f = 0; f < s->nf; ++f) {
        const int64_t o = node_off[f], nn = node_off[f + 1] - o;
        if (nn <= 0) return fail(REVS_ERR_ARG, "feeder %d has no nodes", f);
        for (int64_t i = 0; i < nn; ++i) {
            const int p = parent[o + i];
            if (p >= i || p < -1) return fail(REVS_ERR_ARG, "feeder %d: nodes must be topologically ordered (parent[i] < i)", f);
            if (!(r[o + i] >= 0.0)) return fail(REVS_ERR_ARG, "feeder %d: negative or NaN resistance at node %lld", f, (long long)i);
            cumr[o + i] = (p < 0 ? 0.0 : cumr[o + p]) + r[o + i];
        }
        for (int64_t j = s->off[f]; j < s->off[f + 1]; ++j) {
            if (res_node[j] < 0 || res_node[j] >= nn) return fail(REVS_ERR_ARG, "res_node[%lld] out of range", (long long)j);
            res_p[s->feeders[f].off + (j - s->off[f])] = res_node[j];
        }
    }
    s->net.valid = false;
    s->net.central_valid = false;
    if (s->pool_nodes < (size_t)total) {
        if (s->d_pool_parent) { cudaFree(s->d_pool_parent); cudaFree(s->d_pool_cumr); s->d_pool_parent = nullptr; s->d_pool_cumr = nullptr; }
        CU(dalloc(&s->d_pool_parent, (size_t)total));
        CU(dalloc(&s->d_pool_cumr, (size_t)total));
        s->pool_nodes = (size_t)total;
    }
    if (!s->d_pool_res) CU(dalloc(&s->d_pool_res, (size_t)s->Hp));
    if (!s->d_pool_off) CU(dalloc(&s->d_pool_off, (size_t)s->nf + 1));
    const double th1 = now_ms();
    {
        std::lock_guard<std::mutex> link(upload_mutex(s->device));
        CU(cudaMemcpyAsync(s->d_pool_parent, parent, sizeof(int) * total, cudaMemcpyHostToDevice, s->sU));
        CU(cudaMemcpyAsync(s->d_pool_cumr, cumr.data(), sizeof(double) * total, cudaMemcpyHostToDevice, s->sU));
        CU(cudaMemcpyAsync(s->d_pool_res, res_p.data(), sizeof(int) * s->Hp, cudaMemcpyHostToDevice, s->sU));
        CU(cudaMemcpyAsync(s->d_pool_off, node_off, sizeof(int64_t) * (s->nf + 1), cudaMemcpyHostToDevice, s->sU));
    }
    {
        bool any = false, moved = false;
        for (int f = 0; f < s->nf; ++f) {
            const bool want = s->feeders[f].n > s->newton_min_n || s->roff_alloc[f] < 0;
            if (want != (bool)s->is_newton[f]) { set_newton(s, f, want); moved = true; }
        }
        if (moved) {
            int rc = build_tables(s);
            if (rc) return rc;
        }
        for (int f = 0; f < s->nf; ++f) {
            if (!s->is_newton[f]) continue;
            const int64_t o = node_off[f];
            newton_build_zone((int)(node_off[f + 1] - o), parent + o, r + o, s->feeders[f].n, res_node + s->off[f], s->nt_host[f]);
            any = true;
        }
        if (any || s->n_newton_cols) {
            int rc = rebuild_newton(s);
            if (rc) return rc;
        }
    }
    int max_n = 0;
    for (int f = 0; f < s->nf; ++f) {
        Tree& t = s->trees[f];
        if (t.d_parent && !t.pooled) { cudaFree(t.d_parent); cudaFree(t.d_cumr); cudaFree(t.d_res_node); }
        t.n_nodes = (int)(node_off[f + 1] - node_off[f]);
        t.d_parent = s->d_pool_parent + node_off[f];
        t.d_cumr = s->d_pool_cumr + node_off[f];
        t.d_res_node = s->d_pool_res + s->feeders[f].off;
        t.pooled = true;
        s->sens_set[f] = 1;
        if (!s->is_newton[f] && s->feeders[f].n > max_n) max_n = s->feeders[f].n;
    }
    if (max_n > 0)
    CU(launch_sens_voltage_batched(s->d_feeders, s->nf, max_n, s->d_pool_off, s->d_pool_parent, s->d_pool_cumr,
                                   s->d_pool_res, s->d_Rpool, s->sU));
    s->stats.kernel_launches++;
    s->rn2_valid = false;
    if (s->debug_host)
        fprintf(stderr, "[revs host] set_feeder_trees: checks + cumulative resistances %.3f ms, copies + zone tables + sensitivity launch %.3f ms\n",
                th1 - th0, now_ms() - th1);
    return REVS_OK;
}

int revs_set_homes(revs_solver* s, const double* load, const uint8_t* has_ev, const double* rating,
                   const double* capacity, const double* initial, const int32_t* start, const int32_t* end) {
    if (!s || !load || !has_ev) return fail(REVS_ERR_ARG, "bad arguments");
    const double th0 = now_ms();
    CU(cudaSetDevice(s->device));
    const int64_t H = s->H, Hp = s->Hp;
    // the per-home vectors go through one page-locked staging block in the padded layout, so
    // that every copy is asynchronous and the call synchronises once
    const size_t nd = (size_t)Hp, bytes = nd * (4 * sizeof(double) + 4 * sizeof(int)) + nd;
    if (s->h_homes_bytes < bytes) {
        if (s->h_homes) cudaFreeHost(s->h_homes);
        s->h_homes = nullptr;
        CU(cudaHostAlloc(&s->h_homes, bytes, cudaHostAllocDefault));
        s->h_homes_bytes = bytes;
    }
    double* rt = reinterpret_cast<double*>(s->h_homes);
    double *cp = rt + nd, *in = cp + nd, *ic = in + nd;
    int* st = reinterpret_cast<int*>(ic + nd);
    int *en = st + nd, *nmin = en + nd, *nmax = nmin + nd;
    uint8_t* ev = reinterpret_cast<uint8_t*>(nmax + nd);
    for (size_t i = 0; i < nd; ++i) { rt[i] = 0.0; cp[i] = 1.0; in[i] = 0.0; ic[i] = 0.0; st[i] = en[i] = nmin[i] = nmax[i] = 0; ev[i] = 0; }
    for (int f = 0; f < s->nf; ++f) {
        const int64_t po = s->feeders[f].off - s->off[f];       // padded index = compact index + po
        for (int64_t i = s->off[f]; i < s->off[f + 1]; ++i) {
            if (!has_ev[i]) continue;
            if (!rating || !capacity || !initial || !start || !end) return fail(REVS_ERR_ARG, "EV arrays missing");
            if (!(rating[i] > 0.0) || !(capacity[i] > 0.0)) return fail(REVS_ERR_ARG, "home %lld: rating and capacity must be positive", (long long)i);
            const int64_t p = i + po;
            ev[p] = 1;
            rt[p] = rating[i]; cp[p] = capacity[i]; in[p] = initial[i];
            st[p] = start[i]; en[p] = end[i];
            count_window(rating[i], capacity[i], initial[i], &nmin[p], &nmax[p]);
            ic[p] = -(0.99 * (rating[i] / capacity[i]));
        }
    }
    int rc;
    const double th1 = now_ms();
    std::lock_guard<std::mutex> link(upload_mutex(s->device));     // held until the copies have landed
    const double th2 = now_ms();
    if ((rc = h2d_homes(s, s->d_load, load, s->T))) return rc;
    CU(cudaMemcpyAsync(s->d_has_ev, ev, nd, cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemcpyAsync(s->d_rating, rt, nd * sizeof(double), cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemcpyAsync(s->d_capacity, cp, nd * sizeof(double), cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemcpyAsync(s->d_initial, in, nd * sizeof(double), cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemcpyAsync(s->d_indconst, ic, nd * sizeof(double), cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemcpyAsync(s->d_start, st, nd * sizeof(int), cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemcpyAsync(s->d_end, en, nd * sizeof(int), cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemcpyAsync(s->d_nmin, nmin, nd * sizeof(int), cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemcpyAsync(s->d_nmax, nmax, nd * sizeof(int), cudaMemcpyHostToDevice, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    (void)H;
    if (s->debug_host)
        fprintf(stderr, "[revs host] set_homes: staging %.3f ms, waiting for the link %.3f ms, copies %.3f ms\n", th1 - th0, th2 - th1, now_ms() - th2);
    s->homes_set = true;
    s->net.central_valid = false;
    return REVS_OK;
}

int revs_set_tariff(revs_solver* s, const double* cost) {
    if (!s || !cost) return fail(REVS_ERR_ARG, "bad arguments");
    CU(cudaSetDevice(s->device));
    CU(cudaMemcpy(s->d_cost, cost, sizeof(double) * s->T, cudaMemcpyHostToDevice));
    s->tariff_set = true;
    s->net.central_valid = false;
    return REVS_OK;
}

int revs_admm_begin(revs_solver* s, double kappa, int iter_max, double vset, double vlow, double vhigh) {
    int rc = check_ready(s);
    if (rc) return rc;
    if (!(kappa > 0.0) || iter_max <= 0) return fail(REVS_ERR_ARG, "kappa and iter_max must be positive");
    const double u = vhigh * vhigh - vset * vset, lo = vlow * vlow - vset * vset;
    if (!(u > 0.0) || !(lo <= 0.0))
        return fail(REVS_ERR_ARG, "need vlow <= vset < vhigh (lpsolver.py:185-193 with g >= 0, R >= 0)");
    CU(cudaSetDevice(s->device));
    s->kappa = kappa; s->iter_max = iter_max; s->vset = vset; s->vlow = vlow; s->vhigh = vhigh;
    s->k = 0; s->cur = 0; s->running = true;
    s->net.repaired_valid = false;   // the repaired schedule belongs to the previous run
    s->warm_cls = 0;                 // multipliers start at zero
    s->ws_bound = 0;
    memset(&s->stats, 0, sizeof s->stats);
    const size_t HT = (size_t)s->Hp * s->T * sizeof(double);
    double* zero[] = {s->d_pest, s->d_psch[0], s->d_psch[1], s->d_gamma, s->d_pev, s->d_zt, s->d_lamt, s->d_gt, s->d_vt};
    for (double* p : zero) CU(cudaMemsetAsync(p, 0, HT, s->sU));
    CU(cudaMemsetAsync(s->d_cnt, 0, sizeof(Counters), s->sU));
    CU(cudaMemsetAsync(s->d_wcount, 0, sizeof(int) * s->ncols, s->sU));
    CU(cudaMemsetAsync(s->d_gbf, 0, HT / sizeof(double) * 2, s->sU));
    if (s->diff_cap < iter_max) {
        if (s->d_diff) CU(cudaFree(s->d_diff));
        s->d_diff = nullptr;
        CU(dalloc(&s->d_diff, (size_t)iter_max * s->Hp));
        s->diff_cap = iter_max;
    }
    if (s->comm_world > 1) {
        s->comm_run += 1ull << 20;             // every rank calls revs_admm_begin the same number of times
        CU(cudaMemcpyAsync(s->d_run_seq, &s->comm_run, sizeof(unsigned long long), cudaMemcpyHostToDevice, s->sU));
        CU(cudaMemsetAsync(s->d_comm_timeout, 0, sizeof(int), s->sU));
    }
    CU(cudaEventRecord(s->evT0, s->sU));
    CU(cudaEventRecord(s->evDualDone, s->sU));
    return REVS_OK;
}

namespace {
DualParams dual_params(revs_solver* s) {
    DualParams D{};
    D.g_t = s->d_gt;
    D.p_sch_new = s->d_psch[1];
    D.p_sch_old = s->d_psch[0];
    D.iter = nullptr;
    D.step = s->k;
    D.iter_max = s->iter_max;
    D.err_a = &s->d_cnt->infeasible;
    D.err_b = &s->d_cnt->n_failed;
    D.cond_loop = 0;
    D.use_cond = 0;
    D.partials = s->d_respart;
    D.dsum = s->d_dsum;                        // every dual update of a loop follows a home solve of the same iteration
    D.peer.world = s->comm_world;
    D.peer.rank = s->comm_rank;
    for (int r = 0; r < kMaxPeers; ++r) D.peer.box[r] = s->peer_box[r];
    D.peer.run_seq = s->d_run_seq;
    D.peer.timeout = s->d_comm_timeout;
    D.gamma = s->d_gamma;
    D.p_est = s->d_pest;
    D.z_t = s->d_zt;
    D.g_next = s->d_gt;
    D.gbf_next = s->screen ? s->d_gbf : nullptr;
    D.diff_k = s->d_diff;
    D.res = &s->d_cnt->res;
    D.Hp = (int)s->Hp;
    D.T = s->T;
    D.kappa = s->kappa;
    D.tol = s->tol;
    D.count = (double)s->H * s->T;
    return D;
}

// wait for the enqueued work, collect spans and counters of the run so far
int finish_sync(revs_solver* s, double sums[3]) {
    CU(cudaStreamSynchronize(s->sU));
    CU(cudaStreamSynchronize(s->sH));
    spans_collect(s);
    int rc = check_device_flags(s);
    if (rc == REVS_OK && s->comm_world > 1) {
        int to = 0;
        CU(cudaMemcpy(&to, s->d_comm_timeout, sizeof(int), cudaMemcpyDeviceToHost));
        if (to) rc = fail(REVS_ERR_CUDA, "a peer GPU did not deliver its residual sums within 10 s (rank %d of %d)", s->comm_rank, s->comm_world);
    }
    if (rc) { s->running = false; return rc; }
    s->stats.primal_residual = s->h_cnt->res.primal;
    s->stats.dual_residual = s->h_cnt->res.dual;
    s->stats.qp_newton_iterations = (int64_t)s->h_cnt->newton_its;
    s->stats.qp_flops = (double)s->h_cnt->qp_flops;
    s->stats.qp_columns = (int64_t)s->h_cnt->qp_cols;
    s->stats.max_working_set = s->h_cnt->max_ws;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, s->evT0, s->evT1);
    s->stats.total_ms = ms;
    if (sums) {
        sums[0] = s->h_cnt->res.sum_primal;
        sums[1] = s->h_cnt->res.sum_dual;
        sums[2] = s->comm_world > 1 ? s->h_cnt->res.count : (double)s->H * s->T;
    }
    return REVS_OK;
}

int admm_step_impl(revs_solver* s, double sums[3], bool sync_now) {
    if (!s || !s->running) return fail(REVS_ERR_ARG, "revs_admm_begin has not been called");
    if (s->k >= s->iter_max) return fail(REVS_ERR_ARG, "iter_max iterations already done");
    CU(cudaSetDevice(s->device));

    // consumer side on its own stream: uses P_est[k], P_sch[k], Gamma[k] (lpsolver.py:273)
    cudaStream_t sHome = s->overlap_home ? s->sH : s->sU;   // overlap_home = 0: in line, for an undisturbed kernel time
    CU(cudaStreamWaitEvent(sHome, s->evDualDone, 0));
    HomeParams hp = home_params(s, 0);
    hp.dsum = s->d_dsum;
    hp.first = s->k == 0 ? 1 : 0;
    TimedSpan* sp = span_begin(s, 1, sHome);
    CU(launch_home_solve(hp, sHome));
    span_end(sp, sHome);
    CU(cudaEventRecord(s->evHomeDone, sHome));
    s->stats.kernel_launches++;

    // operator side
    int rc = utility_solve(s, true);
    if (rc) { s->running = false; cudaDeviceSynchronize(); return rc; }

    // fused dual update / residuals / next target
    CU(cudaStreamWaitEvent(s->sU, s->evHomeDone, 0));
    DualParams D = dual_params(s);
    D.p_sch_new = s->d_psch[s->cur ^ 1];
    D.p_sch_old = s->d_psch[s->cur];
    D.diff_k = s->d_diff + (size_t)s->k * s->Hp;
    sp = span_begin(s, 2, s->sU);
    CU(launch_dual_update(D, s->sU));
    span_end(sp, s->sU);
    s->stats.kernel_launches++;
    CU(cudaEventRecord(s->evDualDone, s->sU));
    CU(cudaMemcpyAsync(s->h_cnt, s->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, s->sU));
    CU(cudaEventRecord(s->evT1, s->sU));
    s->cur ^= 1;
    s->k++;
    s->stats.admm_iterations = s->k;
    if (!sync_now) return REVS_OK;       // the next iteration is enqueued behind this one
    return finish_sync(s, sums);
}

// ---- the whole ADMM loop as ONE captured graph whose two loops are decided on the device:
//
//   while (k < iter_max && !converged && !error)            cudaGraphCondTypeWhile, condition set by the last CTA of dual_update_kernel
//       home_solve            (own branch: uses the previous iterates, joins before dual_update)
//       qp_init
//       tree_newton           (zones of the tree-Newton path, if any)
//       while (columns running)                             cudaGraphCondTypeWhile, condition set by round_end_kernel
//           screening pass, work lists, QP classes side by side, round end      (only when some zone has a dense block)
//       dual_update           (k += 1)
//
// Every kernel reads what changes from iteration to iteration (ping-pong side of the schedules, row of diff,
// round number) from device counters, so the bodies are captured once.  Nothing returns to the host until the
// schedule is finished: no round trip per working-set round, no launch latency per kernel.
int capture_loop(revs_solver* s) {
    const int flags = (s->screen ? 1 : 0) | (s->screen_impl << 1) | (s->overlap_home ? 4 : 0) | (s->use_warp_kernel ? 8 : 0) | (s->use_fast ? 16 : 0) | (s->comm_world << 8) | (s->comm_rank << 16) | (dense_cols(s) ? 64 : 0) | (newton_active(s) ? 128 : 0);
    if (s->loop_exec && s->gk_kappa == s->kappa && s->gk_vset == s->vset && s->gk_vhigh == s->vhigh && s->gk_tol == s->tol &&
        s->gk_iter_max == s->iter_max && s->gk_flags == flags)
        return REVS_OK;
    if (s->loop_exec) { cudaGraphExecDestroy(s->loop_exec); s->loop_exec = nullptr; }
    if (s->loop_graph) { cudaGraphDestroy(s->loop_graph); s->loop_graph = nullptr; }
    // function attributes are set outside the capture
    for (int cl = 1; cl < kQpClasses; ++cl) CU(launch_utility_qp(QpParams{}, 0, cl, s->sU));
    CU(qp_warp_prepare());
    CU(screen_prepare());
    CU(screen_tc5_prepare());
    CU(cudaGraphCreate(&s->loop_graph, 0));
    const bool rounds = dense_cols(s) > 0;         // the working-set loop of the dense kernels
    cudaGraphConditionalHandle h_loop, h_round = 0;
    GateCapture gc{};
    CU(cudaGraphConditionalHandleCreate(&h_loop, s->loop_graph, 1, cudaGraphCondAssignDefault));
    if (rounds) {
        CU(cudaGraphConditionalHandleCreate(&h_round, s->loop_graph, 0, cudaGraphCondAssignDefault));
        for (int cl = 2; cl < kQpClasses; ++cl) CU(cudaGraphConditionalHandleCreate(&gc.h[cl], s->loop_graph, 0, cudaGraphCondAssignDefault));
    }
    cudaGraphNodeParams np_loop{};
    np_loop.type = cudaGraphNodeTypeConditional;
    np_loop.conditional.handle = h_loop;
    np_loop.conditional.type = cudaGraphCondTypeWhile;
    np_loop.conditional.size = 1;
    cudaGraphNode_t n_loop;
    CU(cudaGraphAddNode(&n_loop, s->loop_graph, nullptr, 0, &np_loop));
    cudaGraph_t body_loop = np_loop.conditional.phGraph_out[0];

    // ---- body of the ADMM loop
    cudaGraph_t body_round = nullptr;
    CU(cudaStreamBeginCaptureToGraph(s->sU, body_loop, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
    int rc = REVS_OK;
    auto capture_body = [&]() -> int {
        cudaStream_t sHome = s->overlap_home ? s->sH : s->sU;
        if (s->overlap_home) {
            CU(cudaEventRecord(s->evV, s->sU));
            CU(cudaStreamWaitEvent(s->sH, s->evV, 0));
        }
        HomeParams hp = home_params(s, 0);
        hp.p_sch = s->d_psch[0];
        hp.p_sch_new = s->d_psch[1];
        hp.iter = &s->d_cnt->iter;
        hp.dsum = s->d_dsum;
        CU(launch_home_solve(hp, sHome));
        if (s->overlap_home) CU(cudaEventRecord(s->evHomeDone, s->sH));
        QpParams Q = qp_params(s);
        if (rounds) {                                // qp_init_kernel opens the working-set loop
            Q.cond_round = (unsigned long long)h_round;
            Q.use_cond = 1;
        }
        int r = launch_init(s, Q, true, false);
        if (r) return r;
        if (newton_active(s)) {
            const revs_stats keep = s->stats;
            r = launch_newton_stage(s, false);
            s->stats = keep;
            if (r) return r;
        }
        if (rounds) {
            // the working-set while node goes into the graph being captured, after what the stream has enqueued so far
            cudaStreamCaptureStatus st;
            cudaGraph_t g_cap = nullptr;
            const cudaGraphNode_t* deps = nullptr;
            size_t n_deps = 0;
            CU(cudaStreamGetCaptureInfo(s->sU, &st, nullptr, &g_cap, &deps, &n_deps));
            cudaGraphNodeParams np_round{};
            np_round.type = cudaGraphNodeTypeConditional;
            np_round.conditional.handle = h_round;
            np_round.conditional.type = cudaGraphCondTypeWhile;
            np_round.conditional.size = 1;
            cudaGraphNode_t n_round;
            CU(cudaGraphAddNode(&n_round, g_cap, deps, n_deps, &np_round));
            body_round = np_round.conditional.phGraph_out[0];
            CU(cudaStreamUpdateCaptureDependencies(s->sU, &n_round, 1, cudaStreamSetCaptureDependencies));
        }
        if (s->overlap_home) CU(cudaStreamWaitEvent(s->sU, s->evHomeDone, 0));
        DualParams D = dual_params(s);
        D.iter = &s->d_cnt->iter;
        D.cond_loop = (unsigned long long)h_loop;
        D.use_cond = 1;
        CU(launch_dual_update(D, s->sU));
        return REVS_OK;
    };
    rc = capture_body();
    cudaGraph_t got = nullptr;
    cudaError_t ce = cudaStreamEndCapture(s->sU, &got);
    if (rc) return rc;
    if (ce != cudaSuccess) return fail(REVS_ERR_CUDA, "capture of the ADMM loop body failed: %s", cudaGetErrorString(ce));
    if (rounds) {
        // ---- body of the working-set loop
        CU(cudaStreamBeginCaptureToGraph(s->sU, body_round, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
        auto capture_round = [&]() -> int {
            QpParams Q = qp_params(s);
            const revs_stats keep = s->stats;             // launch accounting of a captured run comes from the device counters
            int r = enqueue_round(s, Q, -1, nullptr, nullptr, false, &gc);
            s->stats = keep;
            if (r) return r;
            RoundEndParams E{};
            E.n_running = &s->d_cnt->n_running;
            E.n_failed = &s->d_cnt->n_failed;
            E.infeasible = &s->d_cnt->infeasible;
            E.round_ctr = &s->d_cnt->round;
            E.noconv = &s->d_cnt->noconv;
            E.rounds_total = &s->d_cnt->rounds_total;
            E.round_max = kQpRoundMax;
            E.cond_round = (unsigned long long)h_round;
            E.use_cond = 1;
            CU(launch_round_end(E, s->sU));
            return REVS_OK;
        };
        rc = capture_round();
        ce = cudaStreamEndCapture(s->sU, &got);
        if (rc) return rc;
        if (ce != cudaSuccess) return fail(REVS_ERR_CUDA, "capture of the working-set loop body failed: %s", cudaGetErrorString(ce));
        for (int cl = 2; cl < kQpClasses; ++cl) {          // bodies of the class gates: the CTA kernel of that class
            CU(cudaStreamBeginCaptureToGraph(s->sQ[cl], gc.body[cl], nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
            QpParams Q = qp_params(s);
            cudaError_t le = launch_utility_qp(Q, s->ncols, cl, s->sQ[cl]);
            ce = cudaStreamEndCapture(s->sQ[cl], &got);
            if (le != cudaSuccess || ce != cudaSuccess)
                return fail(REVS_ERR_CUDA, "capture of QP class %d failed: %s", cl, cudaGetErrorString(le != cudaSuccess ? le : ce));
        }
    }
    CU(cudaGraphInstantiate(&s->loop_exec, s->loop_graph, 0));
    s->gk_kappa = s->kappa; s->gk_vset = s->vset; s->gk_vhigh = s->vhigh; s->gk_tol = s->tol;
    s->gk_iter_max = s->iter_max; s->gk_flags = flags;
    return REVS_OK;
}
}  // namespace

int revs_admm_step(revs_solver* s, double sums[3]) { return admm_step_impl(s, sums, true); }

int revs_solve_admm(revs_solver* s, double kappa, int iter_max, double vset, double vlow, double vhigh,
                    double tol, int* iters_done) {
    const double th0 = now_ms();
    int rc = revs_admm_begin(s, kappa, iter_max, vset, vlow, vhigh);
    if (rc) return rc;
    s->host_sync_ms = 0.0;
    for (double& v : s->cat_ms) v = 0.0;
    const double th1 = now_ms();
    s->tol = tol;
    if (s->use_graph) {
        // one graph launch: both loops run on the device (capture_loop)
        if ((rc = prepare_sensitivity(s))) return rc;
        if ((rc = capture_loop(s))) { s->tol = 0.0; return rc; }
        CU(cudaGraphLaunch(s->loop_exec, s->sU));
        CU(cudaMemcpyAsync(s->h_cnt, s->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, s->sU));
        CU(cudaEventRecord(s->evT1, s->sU));
        CU(cudaEventRecord(s->evDualDone, s->sU));
        rc = finish_sync(s, nullptr);
        s->tol = 0.0;
        s->k = s->h_cnt->iter;
        s->cur = s->k & 1;
        s->stats.admm_iterations = s->k;
        s->stats.qp_outer_iterations = (int64_t)s->h_cnt->rounds_total;
        s->stats.gemm_launches = (int64_t)s->h_cnt->rounds_total;
        s->stats.gemm_full_launches = s->k;
        s->stats.qp_warp_rounds = (s->use_warp_kernel && s->zg.warp_n > 0) ? (int64_t)s->h_cnt->rounds_total : 0;
        // per iteration: home solve, qp_init, tree-Newton, dual update; per working-set round: round_launches
        s->stats.kernel_launches += (int64_t)s->k * (newton_active(s) ? 4 : 3) + (int64_t)s->h_cnt->rounds_total * round_launches(s);
        if (rc) return rc;
    } else {
        for (int k = 0; k < iter_max; ++k) {
            // with a fixed iteration count (tol <= 0, the reference's setting) nothing has to come
            // back to the host between iterations
            rc = admm_step_impl(s, nullptr, tol > 0.0 || k == iter_max - 1);
            if (rc) { s->tol = 0.0; return rc; }
            if (tol > 0.0 && s->h_cnt->res.converged) break;
        }
        s->tol = 0.0;
    }
    if (s->debug_host)
        fprintf(stderr, "[revs host] dev %d: begin %.3f ms, loop %.3f ms (waiting in round syncs %.3f ms), device span %.3f ms, %s | "
                "span sums: screen %.2f+%.2f home %.2f dual %.2f cls1 %.2f cls2-3 %.2f init %.2f warp-mid/big %.2f warp-small %.2f\n",
                s->device, th1 - th0, now_ms() - th1, s->host_sync_ms, s->stats.total_ms, s->use_graph ? "captured loop" : "host-driven loop",
                s->cat_ms[5], s->cat_ms[0], s->cat_ms[1], s->cat_ms[2], s->cat_ms[3], s->cat_ms[4], s->cat_ms[6], s->cat_ms[7], s->cat_ms[8]);
    if (iters_done) *iters_done = s->k;
    return REVS_OK;
}

static int get_results_impl(const revs_solver* s, double* P_sch, double* P_ev, double* SOC, double* diff, int diff_rows, int64_t diff_ld) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    if (diff && diff_ld < s->H) return fail(REVS_ERR_ARG, "diff_ld must be at least the number of homes (%lld)", (long long)s->H);
    if (s->k == 0) return fail(REVS_ERR_ARG, "no ADMM iteration has run");
    if (diff && diff_rows < s->k)
        return fail(REVS_ERR_ARG, "diff holds %d rows but %d ADMM iterations have run", diff_rows, s->k);
    CU(cudaSetDevice(s->device));
    int rc;
    if (P_sch && (rc = d2h_homes(s, P_sch, s->d_psch[s->cur], s->T))) return rc;
    if (P_ev && (rc = d2h_homes(s, P_ev, s->d_pev, s->T))) return rc;
    if (SOC) {
        CU(launch_soc_profile(s->d_pev, s->d_has_ev, s->d_capacity, s->d_initial, s->d_soc, (int)s->Hp, s->T, s->sU));
        const_cast<revs_solver*>(s)->stats.kernel_launches++;
        if ((rc = d2h_homes(s, SOC, s->d_soc, s->T + 1))) return rc;
    }
    if (diff && s->H > 0) {
        // all iterations through the staging buffer in as few transfers as it holds (T + 1 rows each)
        const int chunk = s->T + 1;
        for (int k0 = 0; k0 < s->k; k0 += chunk) {
            const int nk = std::min(chunk, s->k - k0);
            for (int k = 0; k < nk; ++k)
                CU(launch_pack_rows(s->d_diff + (size_t)(k0 + k) * s->Hp, s->d_stage + (size_t)k * s->H, s->d_hmap, s->H, 1, 0, s->sU));
            if (diff_ld == s->H)
                CU(cudaMemcpyAsync(diff + (size_t)k0 * s->H, s->d_stage, (size_t)nk * s->H * sizeof(double), cudaMemcpyDeviceToHost, s->sU));
            else      // rows of the caller's array are longer than this solver's homes (a column block of a shared array)
                CU(cudaMemcpy2DAsync(diff + (size_t)k0 * diff_ld, (size_t)diff_ld * sizeof(double), s->d_stage, (size_t)s->H * sizeof(double),
                                     (size_t)s->H * sizeof(double), (size_t)nk, cudaMemcpyDeviceToHost, s->sU));
        }
    }
    CU(cudaStreamSynchronize(s->sU));
    return REVS_OK;
}

int revs_get_results(const revs_solver* s, double* P_sch, double* P_ev, double* SOC, double* diff, int diff_rows) {
    return get_results_impl(s, P_sch, P_ev, SOC, diff, diff_rows, s ? s->H : 0);
}

int revs_get_schedule(const revs_solver* s, double* P_sch, uint64_t* hour_mask, int mask_words, double* diff, int diff_rows) {
    return revs_get_schedule_ld(s, P_sch, hour_mask, mask_words, diff, diff_rows, s ? s->H : 0);
}

int revs_get_schedule_ld(const revs_solver* s, double* P_sch, uint64_t* hour_mask, int mask_words, double* diff, int diff_rows,
                         int64_t diff_ld) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    if (s->k == 0) return fail(REVS_ERR_ARG, "no ADMM iteration has run");
    if (hour_mask && mask_words != (s->T + 63) / 64) return fail(REVS_ERR_ARG, "mask_words must be ceil(T / 64) = %d", (s->T + 63) / 64);
    CU(cudaSetDevice(s->device));
    // P_sch goes with the other results: their gathers are not counted as launches
    int rc = schedule_d2h(s, s->d_psch[s->cur], s->d_pev, nullptr, hour_mask, mask_words,
                          &const_cast<revs_solver*>(s)->stats.kernel_launches);
    if (rc) return rc;
    return get_results_impl(s, P_sch, nullptr, nullptr, diff, diff_rows, diff_ld);
}

int revs_get_estimate(const revs_solver* s, double* P_est, double* Gamma) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    CU(cudaSetDevice(s->device));
    int rc;
    if (P_est && (rc = d2h_homes(s, P_est, s->d_pest, s->T))) return rc;
    if (Gamma && (rc = d2h_homes(s, Gamma, s->d_gamma, s->T))) return rc;
    CU(cudaStreamSynchronize(s->sU));
    return REVS_OK;
}

int revs_solve_individual(revs_solver* s, double* P_res, double* P_ev, double* SOC) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    if (!s->homes_set || !s->tariff_set) return fail(REVS_ERR_ARG, "homes and tariff must be set");
    CU(cudaSetDevice(s->device));
    s->running = false;
    memset(&s->stats, 0, sizeof s->stats);
    CU(cudaMemsetAsync(s->d_cnt, 0, sizeof(Counters), s->sU));
    s->cur = 0;
    HomeParams hp = home_params(s, 1);
    CU(cudaEventRecord(s->evT0, s->sU));
    CU(launch_home_solve(hp, s->sU));
    CU(launch_soc_profile(s->d_pev, s->d_has_ev, s->d_capacity, s->d_initial, s->d_soc, (int)s->Hp, s->T, s->sU));
    CU(cudaEventRecord(s->evT1, s->sU));
    s->stats.kernel_launches = 2;
    int rc;
    if (P_res && (rc = d2h_homes(s, P_res, s->d_psch[1], s->T))) return rc;
    if (P_ev && (rc = d2h_homes(s, P_ev, s->d_pev, s->T))) return rc;
    if (SOC && (rc = d2h_homes(s, SOC, s->d_soc, s->T + 1))) return rc;
    CU(cudaMemcpyAsync(s->h_cnt, s->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    cudaEventElapsedTime(&s->stats.total_ms, s->evT0, s->evT1);
    s->stats.home_ms = s->stats.total_ms;
    if (s->h_cnt->infeasible) return fail(REVS_ERR_INFEASIBLE, "a home charging sub-problem is infeasible");
    return REVS_OK;
}

int revs_home_step(revs_solver* s, double kappa, const double* p_est, const double* p_sch, const double* gamma,
                   double* P_sch_new, double* P_ev) {
    if (!s || !p_est || !p_sch || !gamma) return fail(REVS_ERR_ARG, "bad arguments");
    if (!s->homes_set || !s->tariff_set) return fail(REVS_ERR_ARG, "homes and tariff must be set");
    CU(cudaSetDevice(s->device));
    s->running = false;
    s->kappa = kappa;
    s->cur = 0;
    int rc;
    if ((rc = h2d_homes(s, s->d_pest, p_est, s->T))) return rc;
    if ((rc = h2d_homes(s, s->d_psch[0], p_sch, s->T))) return rc;
    if ((rc = h2d_homes(s, s->d_gamma, gamma, s->T))) return rc;
    CU(cudaMemsetAsync(s->d_cnt, 0, sizeof(Counters), s->sU));
    HomeParams hp = home_params(s, 0);
    CU(launch_home_solve(hp, s->sU));
    s->stats.kernel_launches++;
    if (P_sch_new && (rc = d2h_homes(s, P_sch_new, s->d_psch[1], s->T))) return rc;
    if (P_ev && (rc = d2h_homes(s, P_ev, s->d_pev, s->T))) return rc;
    CU(cudaMemcpyAsync(s->h_cnt, s->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    if (s->h_cnt->infeasible) return fail(REVS_ERR_INFEASIBLE, "a home charging sub-problem is infeasible");
    return REVS_OK;
}

int revs_utility_step(revs_solver* s, double kappa, double vset, double vlow, double vhigh, const double* p_est,
                      const double* p_sch, const double* gamma, const double* lam0, double* P_est_new,
                      double* lam_out) {
    if (!s || !p_est || !p_sch || !gamma) return fail(REVS_ERR_ARG, "bad arguments");
    for (int f = 0; f < s->nf; ++f)
        if (!s->sens_set[f]) return fail(REVS_ERR_ARG, "feeder %d has no sensitivity block", f);
    const double u = vhigh * vhigh - vset * vset, lo = vlow * vlow - vset * vset;
    if (!(u > 0.0) || !(lo <= 0.0) || !(kappa > 0.0))
        return fail(REVS_ERR_ARG, "need kappa > 0 and vlow <= vset < vhigh");
    CU(cudaSetDevice(s->device));
    s->running = false;
    s->kappa = kappa; s->vset = vset; s->vlow = vlow; s->vhigh = vhigh;
    const int T = s->T;
    const size_t HT = (size_t)s->Hp * T;
    std::vector<double> zt(HT, 0.0), lt(HT, 0.0);
    for (int f = 0; f < s->nf; ++f)
        for (int64_t i = s->off[f]; i < s->off[f + 1]; ++i) {
            const int64_t hp = s->feeders[f].off + (i - s->off[f]);
            for (int t = 0; t < T; ++t) {
                const size_t src = (size_t)i * T + t;
                zt[(size_t)t * s->Hp + hp] = (p_est[src] + p_sch[src]) / 2.0 - gamma[src] / kappa;
                // only positive multipliers start a working set (qp_init_kernel): zero, negative and NaN entries are
                // stored as 0, so that no row outside the solution comes back with the caller's value
                if (lam0) lt[(size_t)t * s->Hp + hp] = lam0[src] > 0.0 ? lam0[src] : 0.0;
            }
        }
    CU(cudaMemcpyAsync(s->d_zt, zt.data(), HT * sizeof(double), cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemcpyAsync(s->d_lamt, lt.data(), HT * sizeof(double), cudaMemcpyHostToDevice, s->sU));
    CU(cudaMemsetAsync(s->d_gt, 0, HT * sizeof(double), s->sU));
    CU(cudaMemsetAsync(s->d_vt, 0, HT * sizeof(double), s->sU));
    CU(cudaMemsetAsync(s->d_cnt, 0, sizeof(Counters), s->sU));
    CU(cudaMemsetAsync(s->d_wcount, 0, sizeof(int) * s->ncols, s->sU));
    memset(&s->stats, 0, sizeof s->stats);
    s->warm_cls = kQpClasses - 1;    // caller-supplied multipliers: any class
    s->ws_bound = kWMax;
    int rc = utility_solve(s);
    spans_collect(s);
    if (rc) return rc;
    s->stats.qp_newton_iterations = (int64_t)s->h_cnt->newton_its;
    s->stats.max_working_set = s->h_cnt->max_ws;
    std::vector<double> gt(HT);
    CU(cudaMemcpy(gt.data(), s->d_gt, HT * sizeof(double), cudaMemcpyDeviceToHost));
    if (lam_out) CU(cudaMemcpy(lt.data(), s->d_lamt, HT * sizeof(double), cudaMemcpyDeviceToHost));
    for (int f = 0; f < s->nf; ++f)
        for (int64_t i = s->off[f]; i < s->off[f + 1]; ++i) {
            const int64_t hp = s->feeders[f].off + (i - s->off[f]);
            for (int t = 0; t < T; ++t) {
                if (P_est_new) P_est_new[(size_t)i * T + t] = gt[(size_t)t * s->Hp + hp];
                if (lam_out) lam_out[(size_t)i * T + t] = lt[(size_t)t * s->Hp + hp];
            }
        }
    return REVS_OK;
}

}  // extern "C"

namespace {
// sharded: this rank contracts only its block of the rows; the epilogue stores them into every rank's gather buffer
int reliability_impl(revs_solver* s, int feeder, int kind, int n_rows_all, const int32_t* rows_all, const double* scale_all,
                     double vset, const double* P, double* out, bool sharded) {
    if (!s || feeder < 0 || feeder >= s->nf || n_rows_all < 0 || !rows_all || !out) return fail(REVS_ERR_ARG, "bad arguments");
    int n_rows = n_rows_all, row_lo = 0;
    const int32_t* rows = rows_all;
    const double* scale = scale_all;
    if (sharded) {
        if (s->gather_world < 1 || !s->d_gather) return fail(REVS_ERR_ARG, "call revs_gather_export / revs_gather_attach first");
        if ((int64_t)n_rows_all * s->T > s->gather_cap)
            return fail(REVS_ERR_ARG, "gather buffer holds %lld doubles, %lld needed", (long long)s->gather_cap, (long long)n_rows_all * s->T);
        if (!P) return fail(REVS_ERR_ARG, "the sharded check needs the schedule of the whole feeder on every rank");
        // contiguous blocks of whole contraction tiles, so that no tile straddles two ranks
        const int bm = contract_tile_rows(s->T);
        const int tiles = (n_rows_all + bm - 1) / bm;
        const int t_lo = (int)((int64_t)tiles * s->gather_rank / s->gather_world), t_hi = (int)((int64_t)tiles * (s->gather_rank + 1) / s->gather_world);
        row_lo = std::min(n_rows_all, t_lo * bm);
        n_rows = std::min(n_rows_all, t_hi * bm) - row_lo;
        rows = rows_all + row_lo;
        scale = scale_all ? scale_all + row_lo : nullptr;
    }
    if (kind != REVS_REL_VOLTAGE && kind != REVS_REL_FLOW && kind != REVS_REL_DROP) return fail(REVS_ERR_ARG, "bad kind");
    const Tree& t = s->trees[feeder];
    if (!t.d_parent) return fail(REVS_ERR_ARG, "feeder %d has no tree (call revs_set_feeder_tree)", feeder);
    if (!P && s->k == 0) return fail(REVS_ERR_ARG, "no schedule given and no ADMM result available");
    for (int i = 0; i < n_rows_all; ++i)
        if (rows_all[i] < 0 || rows_all[i] >= t.n_nodes) return fail(REVS_ERR_ARG, "rows[%d] out of range", i);
    if (n_rows_all == 0) return REVS_OK;
    CU(cudaSetDevice(s->device));
    const FeederDev& fd = s->feeders[feeder];
    const int T = s->T;
    int* d_rows = nullptr;
    double *d_S = nullptr, *d_Pt = nullptr, *d_P = nullptr, *d_out = nullptr, *d_scale = nullptr;
    ContractProblem* d_prob = nullptr;
    ContractTile* d_tiles = nullptr;
    int rc = REVS_OK;
    auto cleanup = [&]() {
        cudaFree(d_rows); cudaFree(d_S); cudaFree(d_Pt); cudaFree(d_P); cudaFree(d_out); cudaFree(d_scale);
        cudaFree(d_prob); cudaFree(d_tiles);
    };
#define TRYR(x)                                                                          \
    do {                                                                                 \
        cudaError_t e_ = (x);                                                            \
        if (e_ != cudaSuccess) {                                                         \
            cleanup();                                                                   \
            return fail(REVS_ERR_CUDA, "%s failed: %s", #x, cudaGetErrorString(e_));     \
        }                                                                                \
    } while (0)
    TRYR(dalloc(&d_rows, (size_t)n_rows));
    if (n_rows) TRYR(cudaMemcpy(d_rows, rows, sizeof(int) * n_rows, cudaMemcpyHostToDevice));
    TRYR(dalloc(&d_S, (size_t)n_rows * fd.np));
    TRYR(dalloc(&d_Pt, (size_t)T * fd.np));
    TRYR(dalloc(&d_out, (size_t)n_rows * T));
    const double* src = s->d_psch[s->cur] + (size_t)fd.off * T;
    if (P) {
        TRYR(dalloc(&d_P, (size_t)fd.n * T));
        TRYR(cudaMemcpy(d_P, P, sizeof(double) * fd.n * T, cudaMemcpyHostToDevice));
        src = d_P;
    }
    if (n_rows == 0) {
        // (more ranks than tiles: this rank only signals and waits)
    } else if (kind == REVS_REL_FLOW) {
        TRYR(launch_sens_flow(t.d_parent, d_rows, t.d_res_node, n_rows, fd.n, d_S, fd.np, s->sU));
        if (scale) {
            TRYR(dalloc(&d_scale, (size_t)n_rows));
            TRYR(cudaMemcpy(d_scale, scale, sizeof(double) * n_rows, cudaMemcpyHostToDevice));
        }
    } else {
        TRYR(launch_sens_voltage(t.d_parent, t.d_cumr, d_rows, t.d_res_node, n_rows, fd.n, d_S, fd.np, s->sU));
    }
    TRYR(launch_to_time_major(src, fd.n, T, d_Pt, fd.np, s->sU));
    unsigned long long* my_flags = sharded ? reinterpret_cast<unsigned long long*>(s->d_gather + 2 * s->gather_cap) : nullptr;
    size_t half = 0;           // the payload is double-buffered by the parity of the exchange: a peer may still be reading the last one
    if (sharded) {
        GatherDev G{};
        G.seq = ++s->gather_seq;
        half = (size_t)(G.seq & 1ull) * (size_t)s->gather_cap;
        for (int r = 0; r < s->gather_world; ++r) {
            G.out[r] = s->peer_gather[r] + half;
            G.flag[r] = reinterpret_cast<unsigned long long*>(s->peer_gather[r] + 2 * s->gather_cap);
        }
        G.ticket = s->d_gather_ticket;
        G.world = s->gather_world; G.rank = s->gather_rank;
        G.row_base = row_lo;
        G.ldo = T;
        TRYR(cudaMemcpyAsync(s->d_gather_dev, &G, sizeof G, cudaMemcpyHostToDevice, s->sU));
        TRYR(cudaMemsetAsync(s->d_gather_ticket, 0, sizeof(unsigned), s->sU));
        TRYR(cudaMemsetAsync(s->d_gather_timeout, 0, sizeof(int), s->sU));
    }
    {
        ContractProblem pb{d_S, fd.np, n_rows, fd.np, d_Pt, fd.np, d_out, T, d_scale, nullptr, sharded ? s->d_gather_dev : nullptr};
        std::vector<ContractTile> tiles;
        const int bm = contract_tile_rows(T);
        for (int r0 = 0; r0 < n_rows; r0 += bm) tiles.push_back(ContractTile{0, r0});
        TRYR(dalloc(&d_prob, (size_t)1));
        TRYR(cudaMemcpy(d_prob, &pb, sizeof pb, cudaMemcpyHostToDevice));
        TRYR(dalloc(&d_tiles, tiles.size()));
        if (!tiles.empty()) TRYR(cudaMemcpy(d_tiles, tiles.data(), tiles.size() * sizeof(ContractTile), cudaMemcpyHostToDevice));
        int mode = kind == REVS_REL_VOLTAGE ? kOutVoltage : (kind == REVS_REL_FLOW ? kOutScaled : kOutNodeMajor);
        TRYR(launch_contract(d_prob, d_tiles, (int)tiles.size(), T, mode, vset * vset, s->sU));
    }
    if (sharded) {
        if (n_rows == 0) {
            // nothing contracted here: raise the arrival flags from the host side of this stream
            for (int r = 0; r < s->gather_world; ++r)
                TRYR(cudaMemcpyAsync(reinterpret_cast<unsigned long long*>(s->peer_gather[r] + 2 * s->gather_cap) + s->gather_rank, &s->gather_seq,
                                     sizeof(unsigned long long), cudaMemcpyHostToDevice, s->sU));
        }
        TRYR(launch_gather_wait(my_flags, s->gather_world, s->gather_seq, s->d_gather_timeout, s->sU));
        int to = 0;
        TRYR(cudaMemcpyAsync(&to, s->d_gather_timeout, sizeof(int), cudaMemcpyDeviceToHost, s->sU));
        TRYR(cudaMemcpyAsync(out, s->d_gather + half, sizeof(double) * n_rows_all * T, cudaMemcpyDeviceToHost, s->sU));
        TRYR(cudaStreamSynchronize(s->sU));
        if (to) { cleanup(); return fail(REVS_ERR_CUDA, "a peer GPU did not deliver its rows within 10 s (rank %d of %d)", s->gather_rank, s->gather_world); }
    } else {
        TRYR(cudaMemcpyAsync(out, d_out, sizeof(double) * n_rows * T, cudaMemcpyDeviceToHost, s->sU));
        TRYR(cudaStreamSynchronize(s->sU));
    }
#undef TRYR
    s->stats.kernel_launches += 3 + (sharded ? 1 : 0);
    s->stats.gemm_launches += 1;
    cleanup();
    return rc;
}
}  // namespace

extern "C" {

int revs_reliability(revs_solver* s, int feeder, int kind, int n_rows, const int32_t* rows, const double* scale,
                     double vset, const double* P, double* out) {
    return reliability_impl(s, feeder, kind, n_rows, rows, scale, vset, P, out, false);
}

int revs_reliability_sharded(revs_solver* s, int feeder, int kind, int n_rows, const int32_t* rows, const double* scale,
                             double vset, const double* P, double* out) {
    return reliability_impl(s, feeder, kind, n_rows, rows, scale, vset, P, out, true);
}

}  // extern "C"

namespace {
// The breadth-first arrays of revs_network_check, from the trees on the device (nothing of this runs in
// revs_set_feeder_tree(s), which the schedule path times end to end).
int net_prepare(revs_solver* s) {
    if (s->net.valid) return REVS_OK;
    for (int f = 0; f < s->nf; ++f)
        if (!s->trees[f].d_parent)
            return fail(REVS_ERR_ARG, "zone %d has no tree (given as a sensitivity block): the network check needs "
                        "revs_set_feeder_tree(s)", f);
    NetHost h;
    std::vector<int> par, res;
    std::vector<double> cumr, all_cumr;
    for (int f = 0; f < s->nf; ++f) {
        const Tree& t = s->trees[f];
        const FeederDev& fd = s->feeders[f];
        par.resize(t.n_nodes);
        cumr.resize(t.n_nodes);
        res.resize(fd.n);
        CU(cudaMemcpy(par.data(), t.d_parent, sizeof(int) * t.n_nodes, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(cumr.data(), t.d_cumr, sizeof(double) * t.n_nodes, cudaMemcpyDeviceToHost));
        if (fd.n) CU(cudaMemcpy(res.data(), t.d_res_node, sizeof(int) * fd.n, cudaMemcpyDeviceToHost));
        net_add_zone(h, t.n_nodes, par.data(), cumr.data(), fd.n, res.data(), fd.off);
        all_cumr.insert(all_cumr.end(), cumr.begin(), cumr.end());
    }
    net_finish(h, s->T);
    s->net.bf = NetArrays();     // frees the arrays of the previous trees
    NetArrays& b = s->net.bf;
    CU(b.part.alloc(h.ctas.size()));
    CU(b.sum.alloc((size_t)1));
    CU(b.zw.alloc((size_t)3 * s->nf));
    CU(b.gstate.alloc((size_t)h.gstate_doubles));
    CU(b.zones.upload(h.zones));
    CU(b.cumr.upload(all_cumr));
    CU(b.nodes.upload(h.nodes));
    CU(b.levels.upload(h.levels));
    CU(b.res.upload(h.res));
    CU(b.lists.upload(h.lists));
    CU(b.zone_cta.upload(h.zone_cta));
    CU(b.ctas.upload(h.ctas));
    b.h = std::move(h);
    s->net.valid = true;
    return REVS_OK;
}

// The network check kernels on the schedule P (device, [Hp][T]): per-CTA partials, zone_worst and the summary, and
// optionally the voltages, loadings and residence drops.
int net_run(revs_solver* s, const double* P, double v2, double u, double low, double row_tol, const double* scale,
            double* voltage, double* loading, double* drop, int64_t* launches) {
    const NetArrays& b = s->net.bf;
    const NetHost& h = b.h;
    NetParams prm{};
    prm.zones = b.zones;
    prm.nodes = b.nodes;
    prm.levels = b.levels;
    prm.res = b.res;
    prm.ctas = b.ctas;
    prm.P = P;
    prm.scale = scale;
    prm.voltage = voltage;
    prm.loading = loading;
    prm.drop = drop;
    prm.gstate = b.gstate;
    prm.part = b.part;
    prm.T = s->T;
    prm.v2 = v2;
    prm.u = u;
    prm.low = low;
    prm.row_tol = row_tol;
    for (int c = 0; c < 3; ++c) {
        const int n = h.class_off[c + 1] - h.class_off[c];
        if (n == 0) continue;
        CU(launch_network_check(prm, b.lists + h.class_off[c], n, c == 2 ? 0 : h.class_smem[c], s->sU));
        ++*launches;
    }
    CU(launch_network_reduce(b.part, b.zone_cta, s->nf, b.zw, b.sum, s->sU));
    ++*launches;
    return REVS_OK;
}

// A tool's state besides the zone arrays: [Hp][T] scratch up to the number the tool uses, its kept schedule and per-zone
// buffers, the repair kernel's per-zone state (repair, bracket) and the home -> zone map (bracket, certificate).
int net_alloc(revs_solver* s, NetTool tool) {
    static const int n_scratch[] = {1, 2, 9, 1, 0};
    NetTools& t = s->net;
    if (t.ready[tool]) return REVS_OK;
    const size_t HT = (size_t)s->Hp * s->T, nf = (size_t)s->nf;
    for (int i = 0; i < n_scratch[tool]; ++i)
        if (!t.scratch[i]) CU(t.scratch[i].alloc(HT));
    if (tool == kNetRepair) CU(t.repaired.alloc(HT));
    if (tool == kNetCentral) {
        CU(t.central.alloc(HT));
        CU(t.cen_sums.alloc(3 * nf));
        CU(t.cen_bounds.alloc(2 * nf));
        CU(t.cen_state.alloc(nf));
    }
    if (tool == kNetCertify) {
        CU(t.crt_hpos.alloc((size_t)s->Hp));
        CU(t.crt_cert.alloc(4 * nf));
        CU(t.crt_key.alloc(nf));
    }
    if (tool == kNetHosting) {
        CU(t.hc_uni.alloc(nf * s->T));
        CU(t.hc_counts.alloc(3 * nf));
    }
    if ((tool == kNetRepair || tool == kNetCentral) && !t.rep_gws) {
        std::vector<int64_t> off(nf);
        int64_t g = 0;
        for (size_t f = 0; f < nf; ++f) {
            const size_t b = repair_ws_bytes(s->feeders[f].n, s->T);
            if (s->feeders[f].n > kRepairSmemMaxN) {
                off[f] = g;
                g += (int64_t)b;
            } else {
                off[f] = -1;
                t.rep_smem = std::max(t.rep_smem, b);
            }
        }
        CU(t.info.alloc(9 * nf));
        CU(t.rep_wsoff.upload(off));
        CU(t.rep_gws.alloc((size_t)g));
    }
    if ((tool == kNetCentral || tool == kNetCertify) && !t.hzone) {
        std::vector<int> hz((size_t)s->Hp, -1);
        for (size_t f = 0; f < nf; ++f)
            for (int j = 0; j < s->feeders[f].n; ++j) hz[(size_t)s->feeders[f].off + j] = (int)f;
        CU(t.flag.alloc(1));
        CU(t.hzone.upload(hz));
    }
    t.ready[tool] = true;
    return REVS_OK;
}

// The voltage limits of the repair, the bracket and the certificate: v2 = vset^2, u = vhigh^2 - vset^2.
int tool_limits(double vset, double vhigh, double row_tol, double* v2, double* u) {
    *v2 = vset * vset;
    *u = vhigh * vhigh - *v2;
    if (!(vset < vhigh) || !(*u > 0.0)) return fail(REVS_ERR_ARG, "need vset < vhigh");
    if (!(row_tol >= 0.0)) return fail(REVS_ERR_ARG, "row_tol must be >= 0");
    return REVS_OK;
}

// The repair kernel on the schedule P / p_ev (in place) with the drops D of net_run(P), whose zone_worst it reads.
int run_repair(revs_solver* s, double u, double row_tol, double* D, double* P, double* p_ev, int32_t* info) {
    const NetArrays& b = s->net.bf;
    RepairParams rp{};
    rp.zones = b.zones;
    rp.nodes = b.nodes;
    rp.res = b.res;
    rp.cumr = b.cumr;
    rp.zone_worst = b.zw;
    rp.load = s->d_load;
    rp.rating = s->d_rating;
    rp.cost = s->d_cost;
    rp.start = s->d_start;
    rp.end = s->d_end;
    rp.n_min = s->d_nmin;
    rp.D = D;
    rp.P = P;
    rp.p_ev = p_ev;
    rp.gws = s->net.rep_gws;
    rp.ws_off = s->net.rep_wsoff;
    rp.info = info;
    rp.T = s->T;
    rp.u = u;
    rp.row_tol = row_tol;
    CU(launch_repair(rp, s->nf, s->net.rep_smem, s->sU));
    return REVS_OK;
}

// The checks of a schedule source (REVS_NET_*) of revs_network_check and revs_hosting_capacity.
int net_source_check(const revs_solver* s, int source, const double* P) {
    if (source != REVS_NET_SCHEDULE && source != REVS_NET_ESTIMATE && source != REVS_NET_HOST && source != REVS_NET_REPAIRED &&
        source != REVS_NET_CENTRAL)
        return fail(REVS_ERR_ARG, "unknown source %d (REVS_NET_SCHEDULE, REVS_NET_ESTIMATE, REVS_NET_HOST, REVS_NET_REPAIRED "
                    "or REVS_NET_CENTRAL)", source);
    if (source == REVS_NET_HOST && !P) return fail(REVS_ERR_ARG, "REVS_NET_HOST needs the schedule P");
    if (source == REVS_NET_CENTRAL && !s->net.central_valid)
        return fail(REVS_ERR_ARG, "REVS_NET_CENTRAL: revs_central_bracket has not run since the homes, tariff or trees were set");
    if (source != REVS_NET_HOST && source != REVS_NET_CENTRAL && s->k == 0)
        return fail(REVS_ERR_ARG, "no ADMM iteration has run: there is no %s to check",
                    source == REVS_NET_SCHEDULE ? "schedule" : source == REVS_NET_ESTIMATE ? "estimate" : "repaired schedule");
    if (source == REVS_NET_REPAIRED && !s->net.repaired_valid)
        return fail(REVS_ERR_ARG, "REVS_NET_REPAIRED: revs_repair_schedule has not run since the last ADMM run began");
    return REVS_OK;
}

// The device schedule of a checked source; a host schedule P goes to scratch 0 (one launch).
int net_source(revs_solver* s, int source, const double* P, const double** src, int64_t* launches) {
    *src = source == REVS_NET_SCHEDULE ? s->d_psch[s->cur] : source == REVS_NET_REPAIRED ? s->net.repaired
           : source == REVS_NET_CENTRAL ? s->net.central : s->d_pest;
    if (source == REVS_NET_HOST) {
        int rc = net_alloc(s, kNetHostCheck);
        if (rc || (rc = h2d_homes(s, s->net.scratch[0], P, s->T))) return rc;
        *launches += s->H > 0;
        *src = s->net.scratch[0];
    }
    return REVS_OK;
}

// revs_hosting_capacity's CTAs and per-node {W, N}, once per set of trees (after net_prepare).
int hc_ready(revs_solver* s) {
    NetArrays& b = s->net.bf;
    if (b.hc_ready) return REVS_OK;
    hc_prepare(b.h, s->T, b.hc);
    CU(b.hc_ctas.upload(b.hc.ctas));
    CU(b.hc_lists.upload(b.hc.lists));
    CU(b.hc_zone_cta.upload(b.hc.zone_cta));
    CU(b.hc_wn.upload(b.hc.wn));
    CU(b.hc_gstate.alloc((size_t)b.hc.gstate_doubles));
    CU(b.hc_part.alloc(3 * b.hc.ctas.size()));
    b.hc_ready = true;
    return REVS_OK;
}

void net_location(const NetArg& a, int T, int32_t* zone, int32_t* index, int32_t* step) {
    const bool none = a.loc == INT64_MAX;      // no candidate (no residence at all)
    *zone = none ? -1 : a.zone;
    *index = none ? -1 : (int32_t)(a.loc / T);
    *step = none ? -1 : (int32_t)(a.loc % T);
}
}  // namespace

extern "C" {

int revs_network_check(revs_solver* s, int source, const double* P, double vset, double vlow, double vhigh, double row_tol,
                       const double* scale, double* voltage, double* loading, double* zone_worst,
                       revs_network_summary* summary) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    int rc = net_source_check(s, source, P);
    if (rc) return rc;
    const double v2 = vset * vset, u = vhigh * vhigh - v2, lo = vlow * vlow - v2;
    if (!(u > 0.0) || !(lo <= 0.0)) return fail(REVS_ERR_ARG, "need vlow <= vset < vhigh");
    CU(cudaSetDevice(s->device));
    if ((rc = net_prepare(s))) return rc;
    NetArrays& b = s->net.bf;
    const int T = s->T;
    const size_t out_elems = (size_t)b.h.total_nodes * T;
    int64_t launches = 0;
    const double* src = nullptr;
    if ((rc = net_source(s, source, P, &src, &launches))) return rc;
    if (scale) {
        if (!b.scale) CU(b.scale.alloc((size_t)b.h.total_nodes));
        CU(cudaMemcpyAsync(b.scale, scale, sizeof(double) * b.h.total_nodes, cudaMemcpyHostToDevice, s->sU));
    }
    if (voltage && !b.volt) CU(b.volt.alloc(out_elems));
    if (loading && !b.load) CU(b.load.alloc(out_elems));
    if ((rc = net_run(s, src, v2, u, -lo, row_tol, scale ? b.scale.p : nullptr, voltage ? b.volt.p : nullptr,
                      loading ? b.load.p : nullptr, nullptr, &launches)))
        return rc;
    NetPartial m;
    CU(cudaMemcpyAsync(&m, b.sum, sizeof m, cudaMemcpyDeviceToHost, s->sU));
    if (zone_worst) CU(cudaMemcpyAsync(zone_worst, b.zw, sizeof(double) * 3 * s->nf, cudaMemcpyDeviceToHost, s->sU));
    if (voltage) CU(cudaMemcpyAsync(voltage, b.volt, sizeof(double) * out_elems, cudaMemcpyDeviceToHost, s->sU));
    if (loading) CU(cudaMemcpyAsync(loading, b.load, sizeof(double) * out_elems, cudaMemcpyDeviceToHost, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    s->stats.kernel_launches += launches;
    if (summary) {
        revs_network_summary o{};
        o.drop_max = m.drop.v;
        o.v_min = std::sqrt(v2 - m.drop.v);
        net_location(m.drop, T, &o.drop_zone, &o.drop_node, &o.drop_step);
        o.row_excess_max = m.exc.v;
        net_location(m.exc, T, &o.excess_zone, &o.excess_res, &o.excess_step);
        o.rows_violated = (int64_t)m.rows;
        o.nodes_below_vlow = (int64_t)m.low;
        o.loading_max = m.load.v;
        net_location(m.load, T, &o.loading_zone, &o.loading_node, &o.loading_step);
        o.edges_overloaded = (int64_t)m.over;
        *summary = o;
    }
    return REVS_OK;
}

int revs_repair_schedule(revs_solver* s, double vset, double vhigh, double row_tol, double* P_out, uint64_t* hour_mask,
                         int mask_words, int32_t* zone_info) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    if (s->k == 0) return fail(REVS_ERR_ARG, "no ADMM iteration has run: there is no schedule to repair");
    if (hour_mask && mask_words != (s->T + 63) / 64) return fail(REVS_ERR_ARG, "mask_words must be ceil(T / 64) = %d", (s->T + 63) / 64);
    double v2, u;
    int rc = tool_limits(vset, vhigh, row_tol, &v2, &u);
    if (rc) return rc;
    CU(cudaSetDevice(s->device));
    if ((rc = net_prepare(s)) || (rc = net_alloc(s, kNetRepair))) return rc;
    NetTools& t = s->net;
    const size_t HT = (size_t)s->Hp * s->T;
    double *D = t.scratch[0], *pev = t.scratch[1];
    t.repaired_valid = false;
    int64_t launches = 0;
    CU(cudaMemcpyAsync(t.repaired, s->d_psch[s->cur], HT * sizeof(double), cudaMemcpyDeviceToDevice, s->sU));
    CU(cudaMemcpyAsync(pev, s->d_pev, HT * sizeof(double), cudaMemcpyDeviceToDevice, s->sU));
    // the drops of the schedule at every residence, and which zones violate a row
    if ((rc = net_run(s, s->d_psch[s->cur], v2, u, v2, row_tol, nullptr, nullptr, nullptr, D, &launches))) return rc;
    if ((rc = run_repair(s, u, row_tol, D, t.repaired, pev, t.info))) return rc;
    launches += s->nf > 0;
    if ((rc = schedule_d2h(s, t.repaired, pev, P_out, hour_mask, mask_words, &launches))) return rc;
    if (zone_info && s->nf > 0)
        CU(cudaMemcpyAsync(zone_info, t.info, sizeof(int32_t) * 3 * s->nf, cudaMemcpyDeviceToHost, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    s->stats.kernel_launches += launches;
    t.repaired_valid = true;
    return REVS_OK;
}

int revs_central_bracket(revs_solver* s, double vset, double vhigh, double row_tol, int iters, double* P_out,
                         uint64_t* hour_mask, int mask_words, double* zone_bounds, int32_t* zone_info) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    if (!s->homes_set) return fail(REVS_ERR_ARG, "revs_set_homes has not been called");
    if (!s->tariff_set) return fail(REVS_ERR_ARG, "revs_set_tariff has not been called");
    if (iters < 0) return fail(REVS_ERR_ARG, "iters must be >= 0");
    if (hour_mask && mask_words != (s->T + 63) / 64) return fail(REVS_ERR_ARG, "mask_words must be ceil(T / 64) = %d", (s->T + 63) / 64);
    double v2, u;
    int rc = tool_limits(vset, vhigh, row_tol, &v2, &u);
    if (rc) return rc;
    CU(cudaSetDevice(s->device));
    if ((rc = net_prepare(s)) || (rc = net_alloc(s, kNetCentral))) return rc;
    NetTools& t = s->net;
    const int T = s->T, nf = s->nf;
    const size_t HT = (size_t)s->Hp * T;
    double *y = t.scratch[0], *yb = t.scratch[1], *P = t.scratch[2], *pev = t.scratch[3], *D = t.scratch[4],
           *Drep = t.scratch[5], *pev1 = t.scratch[6], *P2 = t.scratch[7], *pev2 = t.scratch[8], *P1 = t.central;
    t.central_valid = false;
    int64_t launches = 0;
    double *cost1 = t.cen_sums, *cost2 = cost1 + nf, *cmax = cost2 + nf;
    int32_t *info1 = t.info, *info2 = info1 + 3 * nf, *info = info2 + 3 * nf;
    CU(cudaMemsetAsync(y, 0, HT * sizeof(double), s->sU));
    CU(cudaMemsetAsync(yb, 0, HT * sizeof(double), s->sU));
    CU(cudaMemsetAsync(t.flag, 0, sizeof(int), s->sU));
    CenSelectParams sp{};
    sp.zones = t.bf.zones;
    sp.hzone = t.hzone;
    sp.load = s->d_load;
    sp.rating = s->d_rating;
    sp.cost = s->d_cost;
    sp.has_ev = s->d_has_ev;
    sp.start = s->d_start;
    sp.end = s->d_end;
    sp.n_min = s->d_nmin;
    sp.n_max = s->d_nmax;
    sp.P = P;
    sp.p_ev = pev;
    sp.infeasible = t.flag;
    sp.Hp = s->Hp;
    sp.T = T;
    // C_max: the most expensive SOC-feasible schedule
    sp.most_expensive = 1;
    CU(launch_central_select(sp, s->sU));
    CU(launch_central_cost(t.bf.zones, nf, s->d_cost, P, T, cmax, s->sU));
    // first start: the repair of e*(0)
    sp.most_expensive = 0;
    CU(launch_central_select(sp, s->sU));
    if ((rc = net_run(s, P, v2, u, v2, row_tol, nullptr, nullptr, nullptr, D, &launches))) return rc;
    CU(cudaMemcpyAsync(Drep, D, HT * sizeof(double), cudaMemcpyDeviceToDevice, s->sU));
    CU(cudaMemcpyAsync(P1, P, HT * sizeof(double), cudaMemcpyDeviceToDevice, s->sU));
    CU(cudaMemcpyAsync(pev1, pev, HT * sizeof(double), cudaMemcpyDeviceToDevice, s->sU));
    if ((rc = run_repair(s, u, row_tol, Drep, P1, pev1, info1))) return rc;
    CU(launch_central_cost(t.bf.zones, nf, s->d_cost, P1, T, cost1, s->sU));
    // the ascent (a host loop: every evaluation is two network checks, the selection and the ascent kernel)
    CenAscentParams ap{};
    ap.zones = t.bf.zones;
    ap.cost = s->d_cost;
    ap.P = P;
    ap.D = D;
    ap.y = y;
    ap.ybest = yb;
    ap.cost1 = cost1;
    ap.cmax = cmax;
    ap.info1 = info1;
    ap.state = t.cen_state;
    ap.iters = iters;
    ap.T = T;
    ap.u = u;
    sp.ry = D;
    for (int k = 0; k <= iters; ++k) {
        if (k > 0) {
            if ((rc = net_run(s, y, v2, u, v2, row_tol, nullptr, nullptr, nullptr, D, &launches))) return rc;
            CU(launch_central_select(sp, s->sU));
            if ((rc = net_run(s, P, v2, u, v2, row_tol, nullptr, nullptr, nullptr, D, &launches))) return rc;
            launches += 1;
        }
        ap.k = k;
        CU(launch_central_ascent(ap, nf, s->sU));
        launches += nf > 0;
    }
    // second start: the repair of e*(y_best)
    if ((rc = net_run(s, yb, v2, u, v2, row_tol, nullptr, nullptr, nullptr, D, &launches))) return rc;
    sp.P = P2;
    sp.p_ev = pev2;
    CU(launch_central_select(sp, s->sU));
    if ((rc = net_run(s, P2, v2, u, v2, row_tol, nullptr, nullptr, nullptr, Drep, &launches))) return rc;
    if ((rc = run_repair(s, u, row_tol, Drep, P2, pev2, info2))) return rc;
    CU(launch_central_cost(t.bf.zones, nf, s->d_cost, P2, T, cost2, s->sU));
    CenFinalParams fp{};
    fp.zones = t.bf.zones;
    fp.state = t.cen_state;
    fp.cost1 = cost1;
    fp.cost2 = cost2;
    fp.cmax = cmax;
    fp.info1 = info1;
    fp.info2 = info2;
    fp.P1 = P1;
    fp.p_ev1 = pev1;
    fp.P2 = P2;
    fp.p_ev2 = pev2;
    fp.bounds = t.cen_bounds;
    fp.info = info;
    fp.T = T;
    CU(launch_central_final(fp, nf, s->sU));
    launches += (s->H > 0 ? 3 : 0) + (nf > 0 ? 6 : 0);     // selections; costs, repairs, final
    int infeasible = 0;
    CU(cudaMemcpyAsync(&infeasible, t.flag, sizeof(int), cudaMemcpyDeviceToHost, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    s->stats.kernel_launches += launches;
    if (infeasible) return fail(REVS_ERR_INFEASIBLE, "a home's SOC target needs more hours than its plug-in window has");
    if ((rc = schedule_d2h(s, P1, pev1, P_out, hour_mask, mask_words, &s->stats.kernel_launches))) return rc;
    if (zone_bounds && nf > 0)
        CU(cudaMemcpyAsync(zone_bounds, t.cen_bounds, sizeof(double) * 2 * nf, cudaMemcpyDeviceToHost, s->sU));
    if (zone_info && nf > 0) CU(cudaMemcpyAsync(zone_info, info, sizeof(int32_t) * 3 * nf, cudaMemcpyDeviceToHost, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    t.central_valid = true;
    return REVS_OK;
}

int revs_certify_infeasible(revs_solver* s, double vset, double vhigh, double row_tol, int32_t* zone_cert,
                            int* n_certified) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    if (!s->homes_set) return fail(REVS_ERR_ARG, "revs_set_homes has not been called");
    double v2, u;
    int rc = tool_limits(vset, vhigh, row_tol, &v2, &u);
    if (rc) return rc;
    CU(cudaSetDevice(s->device));
    if ((rc = net_prepare(s)) || (rc = net_alloc(s, kNetCertify))) return rc;
    const NetTools& t = s->net;
    const int T = s->T, nf = s->nf;
    int64_t launches = 0;
    CU(cudaMemsetAsync(t.flag, 0, sizeof(int), s->sU));
    // the drops of the base load at every residence
    if ((rc = net_run(s, s->d_load, v2, u, v2, row_tol, nullptr, nullptr, nullptr, t.scratch[0], &launches))) return rc;
    CertParams cp{};
    cp.zones = t.bf.zones;
    cp.nodes = t.bf.nodes;
    cp.res = t.bf.res;
    cp.cumr = t.bf.cumr;
    cp.hzone = t.hzone;
    cp.D = t.scratch[0];
    cp.rating = s->d_rating;
    cp.has_ev = s->d_has_ev;
    cp.start = s->d_start;
    cp.end = s->d_end;
    cp.n_min = s->d_nmin;
    cp.n_max = s->d_nmax;
    cp.hpos = t.crt_hpos;
    cp.key = t.crt_key;
    cp.cert = t.crt_cert;
    cp.flag = t.flag;
    cp.Hp = s->Hp;
    cp.T = T;
    cp.u = u;
    cp.thr = row_tol + 1e-12;
    CU(launch_certify(cp, nf, s->sU));
    launches += nf > 0 ? 3 : 0;
    int flag = 0;
    std::vector<int32_t> cert((size_t)4 * nf);
    CU(cudaMemcpyAsync(&flag, t.flag, sizeof(int), cudaMemcpyDeviceToHost, s->sU));
    if (nf > 0) CU(cudaMemcpyAsync(cert.data(), t.crt_cert, sizeof(int32_t) * cert.size(), cudaMemcpyDeviceToHost, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    s->stats.kernel_launches += launches;
    if (flag & 2) return fail(REVS_ERR_ARG, "an EV home has a negative or non-finite rating: the certificate needs rating >= 0");
    if (flag & 1) return fail(REVS_ERR_INFEASIBLE, "a home's SOC target needs more hours than its plug-in window has");
    if (zone_cert && nf > 0) memcpy(zone_cert, cert.data(), sizeof(int32_t) * cert.size());
    if (n_certified) {
        int c = 0;
        for (int f = 0; f < nf; ++f) c += cert[4 * (size_t)f] != 0;
        *n_certified = c;
    }
    return REVS_OK;
}

int revs_hosting_capacity(revs_solver* s, int source, const double* P, double vset, double vhigh, double row_tol,
                          const double* scale, double* home_cap, double* zone_uniform, int64_t* zone_counts) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    int rc = net_source_check(s, source, P);
    if (rc) return rc;
    double v2, u;
    if ((rc = tool_limits(vset, vhigh, row_tol, &v2, &u))) return rc;
    CU(cudaSetDevice(s->device));
    if ((rc = net_prepare(s)) || (rc = net_alloc(s, kNetHosting)) || (rc = hc_ready(s))) return rc;
    NetTools& t = s->net;
    NetArrays& b = t.bf;
    const int T = s->T, nf = s->nf;
    const int64_t N = b.h.total_nodes;
    if (scale)
        for (int64_t i = 0; i < N; ++i)
            if (!std::isfinite(scale[i])) return fail(REVS_ERR_ARG, "scale[%lld] is not finite", (long long)i);
    int64_t launches = 0;
    const double* src = nullptr;
    if ((rc = net_source(s, source, P, &src, &launches))) return rc;
    if (scale) {
        if (!b.scale) CU(b.scale.alloc((size_t)N));
        CU(cudaMemcpyAsync(b.scale, scale, sizeof(double) * N, cudaMemcpyHostToDevice, s->sU));
    }
    if (home_cap && !t.hc_cap) CU(t.hc_cap.alloc((size_t)s->Hp * T));
    HcParams hp{};
    hp.zones = b.zones;
    hp.nodes = b.nodes;
    hp.levels = b.levels;
    hp.res = b.res;
    hp.ctas = b.hc_ctas;
    hp.cumr = b.cumr;
    hp.wn = b.hc_wn;
    hp.P = src;
    hp.scale = scale ? b.scale.p : nullptr;
    hp.has_ev = s->d_has_ev;
    hp.rating = s->d_rating;
    hp.start = s->d_start;
    hp.end = s->d_end;
    hp.cap = home_cap ? t.hc_cap.p : nullptr;
    hp.uniform = t.hc_uni;
    hp.gstate = b.hc_gstate;
    hp.part = b.hc_part;
    hp.T = T;
    hp.ur = u + row_tol;
    const HcHost& h = b.hc;
    for (int c = 0; c < 3; ++c) {
        const int n = h.class_off[c + 1] - h.class_off[c];
        if (n == 0) continue;
        CU(launch_hosting(hp, b.hc_lists + h.class_off[c], n, h.class_smem[c], s->sU));
        ++launches;
    }
    CU(launch_hosting_reduce(b.hc_part, b.hc_zone_cta, nf, t.hc_counts, s->sU));
    launches += nf > 0;
    if (home_cap) {
        if ((rc = d2h_homes(s, home_cap, t.hc_cap, T))) return rc;
        launches += s->H > 0;
    }
    if (zone_uniform && nf > 0)
        CU(cudaMemcpyAsync(zone_uniform, t.hc_uni, sizeof(double) * nf * T, cudaMemcpyDeviceToHost, s->sU));
    if (zone_counts && nf > 0)
        CU(cudaMemcpyAsync(zone_counts, t.hc_counts, sizeof(int64_t) * 3 * nf, cudaMemcpyDeviceToHost, s->sU));
    CU(cudaStreamSynchronize(s->sU));
    s->stats.kernel_launches += launches;
    return REVS_OK;
}

int revs_gather_export(revs_solver* s, int64_t capacity_doubles, void* handle64) {
    if (!s || !handle64 || capacity_doubles <= 0) return fail(REVS_ERR_ARG, "bad arguments");
    CU(cudaSetDevice(s->device));
    for (int r = 0; r < kGatherMaxPeers; ++r) {
        if (s->peer_gather[r] && s->peer_gather[r] != s->d_gather) cudaIpcCloseMemHandle(s->peer_gather[r]);
        s->peer_gather[r] = nullptr;
    }
    if (s->d_gather) { cudaFree(s->d_gather); s->d_gather = nullptr; }
    // two payload halves (alternating exchanges) + arrival flags in one allocation (one IPC handle); cudaMalloc'ed memory is what cudaIpcGetMemHandle exports
    const size_t bytes = (size_t)2 * capacity_doubles * sizeof(double) + kGatherMaxPeers * sizeof(unsigned long long);
    CU(cudaMalloc(&s->d_gather, bytes));
    CU(cudaMemset(s->d_gather, 0, bytes));
    s->gather_cap = capacity_doubles;
    if (!s->d_gather_dev) {
        CU(dalloc(&s->d_gather_dev, (size_t)1));
        CU(dalloc(&s->d_gather_ticket, (size_t)1));
        CU(dalloc(&s->d_gather_timeout, (size_t)1));
    }
    s->gather_world = 1; s->gather_rank = 0; s->gather_seq = 0;
    s->peer_gather[0] = s->d_gather;
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, s->d_gather));
    memcpy(handle64, &h, sizeof h);
    return REVS_OK;
}

int revs_gather_attach(revs_solver* s, int world, int rank, const void* handles) {
    if (!s || !handles || world < 1 || world > kGatherMaxPeers || rank < 0 || rank >= world)
        return fail(REVS_ERR_ARG, "bad arguments (world 1..%d)", kGatherMaxPeers);
    if (!s->d_gather) return fail(REVS_ERR_ARG, "call revs_gather_export first");
    CU(cudaSetDevice(s->device));
    for (int r = 0; r < kGatherMaxPeers; ++r) s->peer_gather[r] = nullptr;
    for (int r = 0; r < world; ++r) {
        if (r == rank) { s->peer_gather[r] = s->d_gather; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles + (size_t)r * sizeof h, sizeof h);
        void* ptr = nullptr;
        CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        s->peer_gather[r] = reinterpret_cast<double*>(ptr);
    }
    s->gather_world = world;
    s->gather_rank = rank;
    s->gather_seq = 0;
    return REVS_OK;
}

int revs_contract(int device, int M, int K, int T, const double* A, const double* B, double* C) {
    if (M <= 0 || K <= 0 || T <= 0 || !A || !B || !C) return fail(REVS_ERR_ARG, "bad arguments");
    int rc = use_device(device);
    if (rc) return rc;
    const int Kp = (K + kPad - 1) / kPad * kPad;
    std::vector<double> Ap((size_t)M * Kp, 0.0), Bt((size_t)T * Kp, 0.0);
    for (int i = 0; i < M; ++i) memcpy(&Ap[(size_t)i * Kp], A + (size_t)i * K, sizeof(double) * K);
    for (int k = 0; k < K; ++k)
        for (int t = 0; t < T; ++t) Bt[(size_t)t * Kp + k] = B[(size_t)k * T + t];
    double *dA = nullptr, *dB = nullptr, *dC = nullptr;
    ContractProblem* d_prob = nullptr;
    ContractTile* d_tiles = nullptr;
    auto cleanup = [&]() { cudaFree(dA); cudaFree(dB); cudaFree(dC); cudaFree(d_prob); cudaFree(d_tiles); };
#define TRYC(x)                                                                          \
    do {                                                                                 \
        cudaError_t e_ = (x);                                                            \
        if (e_ != cudaSuccess) {                                                         \
            cleanup();                                                                   \
            return fail(REVS_ERR_CUDA, "%s failed: %s", #x, cudaGetErrorString(e_));     \
        }                                                                                \
    } while (0)
    TRYC(dalloc(&dA, Ap.size()));
    TRYC(dalloc(&dB, Bt.size()));
    TRYC(dalloc(&dC, (size_t)M * T));
    TRYC(cudaMemcpy(dA, Ap.data(), Ap.size() * sizeof(double), cudaMemcpyHostToDevice));
    TRYC(cudaMemcpy(dB, Bt.data(), Bt.size() * sizeof(double), cudaMemcpyHostToDevice));
    ContractProblem pb{dA, Kp, M, Kp, dB, Kp, dC, T, nullptr, nullptr};
    std::vector<ContractTile> tiles;
    const int bm = contract_tile_rows(T);
    for (int r0 = 0; r0 < M; r0 += bm) tiles.push_back(ContractTile{0, r0});
    TRYC(dalloc(&d_prob, (size_t)1));
    TRYC(cudaMemcpy(d_prob, &pb, sizeof pb, cudaMemcpyHostToDevice));
    TRYC(dalloc(&d_tiles, tiles.size()));
    TRYC(cudaMemcpy(d_tiles, tiles.data(), tiles.size() * sizeof(ContractTile), cudaMemcpyHostToDevice));
    TRYC(launch_contract(d_prob, d_tiles, (int)tiles.size(), T, kOutNodeMajor, 0.0, 0));
    TRYC(cudaMemcpy(C, dC, sizeof(double) * M * T, cudaMemcpyDeviceToHost));
#undef TRYC
    cleanup();
    return REVS_OK;
}

int revs_screen_contract(int device, int M, int K, int T, const double* A, const double* B, double* C, int impl) {
    if (M <= 0 || K <= 0 || T <= 0 || !A || !B || !C) return fail(REVS_ERR_ARG, "bad arguments");
    int rc = use_device(device);
    if (rc) return rc;
    const int Kp = (K + kPad - 1) / kPad * kPad;
    std::vector<double> Ap((size_t)M * Kp, 0.0), Bt((size_t)T * Kp, 0.0);
    for (int i = 0; i < M; ++i) memcpy(&Ap[(size_t)i * Kp], A + (size_t)i * K, sizeof(double) * K);
    for (int k = 0; k < K; ++k)
        for (int t = 0; t < T; ++t) Bt[(size_t)t * Kp + k] = B[(size_t)k * T + t];
    double *dA = nullptr, *dB = nullptr;
    void *dAb = nullptr, *dBb = nullptr, *dmaps = nullptr;
    float* dC = nullptr;
    int* dcol = nullptr;
    ScreenProblem* d_prob = nullptr;
    ContractTile* d_tiles = nullptr;
    auto cleanup = [&]() { cudaFree(dA); cudaFree(dB); cudaFree(dAb); cudaFree(dBb); cudaFree(dC); cudaFree(d_prob); cudaFree(d_tiles); cudaFree(dmaps); cudaFree(dcol); };
#define TRYS(x)                                                                          \
    do {                                                                                 \
        cudaError_t e_ = (x);                                                            \
        if (e_ != cudaSuccess) {                                                         \
            cleanup();                                                                   \
            return fail(REVS_ERR_CUDA, "%s failed: %s", #x, cudaGetErrorString(e_));     \
        }                                                                                \
    } while (0)
    TRYS(dalloc(&dA, Ap.size()));
    TRYS(dalloc(&dB, Bt.size()));
    TRYS(cudaMalloc(&dAb, Ap.size() * 2));
    TRYS(cudaMalloc(&dBb, Bt.size() * 2));
    TRYS(dalloc(&dC, (size_t)M * T));
    TRYS(cudaMemcpy(dA, Ap.data(), Ap.size() * sizeof(double), cudaMemcpyHostToDevice));
    TRYS(cudaMemcpy(dB, Bt.data(), Bt.size() * sizeof(double), cudaMemcpyHostToDevice));
    TRYS(launch_to_bf16(dA, dAb, Ap.size(), 0));
    TRYS(launch_to_bf16(dB, dBb, Bt.size(), 0));
    ScreenProblem pb{dAb, Kp, M, Kp, dBb, Kp, dC, M, nullptr, nullptr};
    std::vector<ContractTile> tiles;
    for (int r0 = 0; r0 < M; r0 += screen_tile_rows()) tiles.push_back(ContractTile{0, r0});
    TRYS(dalloc(&d_prob, (size_t)1));
    TRYS(cudaMemcpy(d_prob, &pb, sizeof pb, cudaMemcpyHostToDevice));
    TRYS(dalloc(&d_tiles, tiles.size()));
    TRYS(cudaMemcpy(d_tiles, tiles.data(), tiles.size() * sizeof(ContractTile), cudaMemcpyHostToDevice));
    if (impl == 1) {
        if (T > (int)screen_tc5_box_rows_b()) { cleanup(); return fail(REVS_ERR_ARG, "tcgen05 screening kernel handles T <= 96"); }
        const size_t mb = screen_tc5_map_bytes();
        std::vector<unsigned char> maps(2 * mb);
        TRYS(screen_tc5_encode(maps.data(), dAb, M, Kp, Kp, screen_tc5_box_rows_a()));
        TRYS(screen_tc5_encode(maps.data() + mb, dBb, T, Kp, Kp, screen_tc5_box_rows_b()));
        TRYS(cudaMalloc(&dmaps, maps.size()));
        TRYS(cudaMemcpy(dmaps, maps.data(), maps.size(), cudaMemcpyHostToDevice));
        TRYS(dalloc(&dcol, (size_t)1));
        TRYS(launch_screen_tc5(d_prob, d_tiles, (int)tiles.size(), dmaps, (const char*)dmaps + mb, dcol, T, 0.0, 0));
    } else {
        TRYS(launch_screen(d_prob, d_tiles, (int)tiles.size(), T, 0.0, 0));
    }
    std::vector<float> out((size_t)M * T);
    TRYS(cudaMemcpy(out.data(), dC, out.size() * sizeof(float), cudaMemcpyDeviceToHost));
#undef TRYS
    for (int i = 0; i < M; ++i)
        for (int t = 0; t < T; ++t) C[(size_t)i * T + t] = (double)out[(size_t)t * M + i];
    cleanup();
    return REVS_OK;
}

int revs_comm_export(revs_solver* s, void* handle64) {
    if (!s || !handle64) return fail(REVS_ERR_ARG, "bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CU(cudaSetDevice(s->device));
    if (!s->d_mailbox) {
        CU(dalloc(&s->d_mailbox, (size_t)2 * kMaxPeers));
        CU(dalloc(&s->d_run_seq, (size_t)1));
        CU(dalloc(&s->d_comm_timeout, (size_t)1));
    }
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, s->d_mailbox));
    memcpy(handle64, &h, sizeof h);
    return REVS_OK;
}

int revs_comm_attach(revs_solver* s, int world, int rank, const void* handles) {
    if (!s || !handles || world < 1 || world > kMaxPeers || rank < 0 || rank >= world)
        return fail(REVS_ERR_ARG, "bad arguments (world 1..%d)", kMaxPeers);
    if (!s->d_mailbox) return fail(REVS_ERR_ARG, "call revs_comm_export first");
    CU(cudaSetDevice(s->device));
    int rc = revs_comm_detach(s);
    if (rc) return rc;
    for (int r = 0; r < world; ++r) {
        if (r == rank) { s->peer_box[r] = s->d_mailbox; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles + (size_t)r * sizeof h, sizeof h);
        void* ptr = nullptr;
        CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        s->peer_box[r] = reinterpret_cast<PeerSlot*>(ptr);
    }
    CU(cudaMemset(s->d_mailbox, 0, sizeof(PeerSlot) * 2 * kMaxPeers));
    s->comm_world = world;
    s->comm_rank = rank;
    s->comm_run = 0;
    return REVS_OK;
}

int revs_comm_detach(revs_solver* s) {
    if (!s) return fail(REVS_ERR_ARG, "null solver");
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->sU));
    for (int r = 0; r < kMaxPeers; ++r) {
        if (s->peer_box[r] && s->peer_box[r] != s->d_mailbox) CU(cudaIpcCloseMemHandle(s->peer_box[r]));
        s->peer_box[r] = nullptr;
    }
    s->comm_world = 1;
    s->comm_rank = 0;
    return REVS_OK;
}

int revs_set_option(revs_solver* s, const char* name, double value) {
    if (!s || !name) return fail(REVS_ERR_ARG, "bad arguments");
    const bool mid_run = s->running && s->k > 0 && s->k < s->iter_max;
    if (!strcmp(name, "screen")) {
        // the error bound of the BF16 screening pass (kScreenUp) holds up to kScreenMaxN residences per zone, and the
        // bf16 copy of the iterate is only maintained while screening is on
        if (value != 0.0 && s->zg.max_n > kScreenMaxN)
            return fail(REVS_ERR_ARG, "screening is limited to zones of at most %d residences", kScreenMaxN);
        if (mid_run) return fail(REVS_ERR_ARG, "'screen' cannot change between revs_admm_step calls of one run");
        s->screen = value != 0.0;
        return REVS_OK;
    }
    if (!strcmp(name, "newton_min_n")) {
        // zones with more residences than this run on their tree (tree_newton.cu: no dense block, any number of binding
        // rows); the default is 512.  Zones above 2048 residences never get a dense block.  Set it before the feeders are given.
        for (int f = 0; f < s->nf; ++f)
            if (s->sens_set[f]) return fail(REVS_ERR_ARG, "set option 'newton_min_n' before the feeders are given");
        s->newton_min_n = value < 0.0 ? 0 : (value > 2e9 ? 2000000000 : (int)value);
        return REVS_OK;
    }
    if (!strcmp(name, "graph")) { s->use_graph = value != 0.0; return REVS_OK; }   // 0: host-driven loop with per-kernel event spans (profiling)
    if (!strcmp(name, "warp_kernel")) { s->use_warp_kernel = value != 0.0; return REVS_OK; }
    if (!strcmp(name, "overlap_home")) { s->overlap_home = value != 0.0; return REVS_OK; }
    if (!strcmp(name, "priority")) {
        // rank of this solver among several on one GPU (0 = served first): its utility streams are
        // re-created `value` levels below the highest stream priority, still above every home solve
        CU(cudaSetDevice(s->device));
        CU(cudaStreamSynchronize(s->sU));
        int pr = s->prio_hi + (int)value;
        if (pr > s->prio_lo - 1) pr = s->prio_lo - 1;
        if (pr < s->prio_hi) pr = s->prio_hi;
        CU(cudaStreamDestroy(s->sU));
        CU(cudaStreamCreateWithPriority(&s->sU, cudaStreamNonBlocking, pr));
        for (int cl = 0; cl < kQpClasses; ++cl) {
            CU(cudaStreamSynchronize(s->sQ[cl]));
            CU(cudaStreamDestroy(s->sQ[cl]));
            CU(cudaStreamCreateWithPriority(&s->sQ[cl], cudaStreamNonBlocking, pr));
        }
        return REVS_OK;
    }
    if (!strcmp(name, "screen_impl")) {
        if (value != 0.0 && !s->tc5_ready) return fail(REVS_ERR_ARG, "tcgen05 screening kernel unavailable (T > 96 or tensor-map encoding failed)");
        s->screen_impl = value != 0.0 ? 1 : 0;
        return REVS_OK;
    }
    return fail(REVS_ERR_ARG, "unknown option '%s'", name);
}

int revs_get_stats(const revs_solver* s, revs_stats* out) {
    if (!s || !out) return fail(REVS_ERR_ARG, "bad arguments");
    *out = s->stats;
    return REVS_OK;
}

}  // extern "C"
