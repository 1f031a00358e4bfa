// Parameter blocks and launchers of the REVS ADMM kernels (one .cu per kernel family).
#pragma once
#include <vector>

#include "common.cuh"

namespace revs {

// ---- home_solve.cu
struct HomeParams {
    const double* load;       // [Hp][T]
    const double* p_est;      // [Hp][T]  previous utility estimate
    const double* p_sch;      // [Hp][T]  previous schedule ...
    const int* iter;          // ... optional device iteration counter k of the ADMM loop: the schedules ping-pong, odd k reads
                              //     p_sch_new and writes p_sch (so one captured launch serves every iteration)
    const double* gamma;      // [Hp][T]
    const double* cost;       // [T]
    const uint8_t* has_ev;    // [Hp]
    const double* rating;     // [Hp]
    const int* start;         // [Hp]
    const int* end;           // [Hp]
    const int* n_min;         // [Hp]  from the SOC rows, host-computed
    const int* n_max;         // [Hp]
    double* p_sch_new;        // [Hp][T]  (const-cast of p_sch is written instead when *iter is odd)
    double* p_ev;             // [Hp][T]
    double* dsum;             // optional [Hp] out: sum over the hours of (new schedule - previous schedule)^2 (dual residual of the ADMM loop)
    int first;                // without `iter`: 1 when the previous schedule is the zero start of the loop (lpsolver.py:250)
    int* infeasible;          // flag
    int Hp, T;
    double kappa;
    int individual;           // 1: objective of solve_residence instead of Home
    const double* ind_const;  // [Hp]  -(0.99*(rating/capacity)), individual mode only
};

cudaError_t launch_home_solve(const HomeParams& P, cudaStream_t stream);
cudaError_t launch_soc_profile(const double* p_ev, const uint8_t* has_ev, const double* capacity,
                               const double* initial, double* soc, int Hp, int T, cudaStream_t stream);

// ---- dual_update.cu
struct ResidualOut {
    double sum_primal;     // sum (P_est - P_sch)^2        (this device, last iteration)
    double sum_dual;       // sum (P_sch - P_sch_prev)^2
    double primal;         // sqrt(sum_primal / count)
    double dual;           // kappa * sqrt(sum_dual / count)
    double count;          // home-hours the sums run over (all ranks when peers are attached)
    int converged;
    unsigned ticket;
};

// All-reduce of the residual sums over the GPUs of one box, done by the last CTA of dual_update_kernel itself
// through peer-mapped mailboxes (NVLink P2P stores + system-scope release/acquire flags): every rank pushes
// {sum primal, sum dual, home-hours} into its slot of every peer's mailbox, then collects the slots of its own
// mailbox in rank order -- the same additions in the same order on every rank, so all ranks take the same
// convergence decision, and the exchange needs no extra launch and works inside the captured loop.
constexpr int kMaxPeers = 16;
struct PeerSlot { double v[3]; unsigned long long seq; };     // 32 bytes; seq = run sequence + iteration + 1
struct PeerReduce {
    int world, rank;                          // world <= 1: off
    PeerSlot* box[kMaxPeers];                 // box[r]: mailbox on GPU r, [2 parities][world slots]; box[rank] is local
    const unsigned long long* run_seq;        // device word, changed by every revs_admm_begin (stale slots never match)
    int* timeout;                             // set when a peer did not show up within ~10 s
};

struct DualParams {
    const double* g_t;         // [T][Hp]  P_est[k+1], time-major (utility output)
    const double* p_sch_new;   // [Hp][T]  (swapped with p_sch_old when *iter is odd)
    const double* p_sch_old;   // [Hp][T]
    const double* dsum;        // optional [Hp]: sum over the hours of (P_sch[k+1] - P_sch[k])^2 per home, left by home_solve_kernel;
                               //     p_sch_old is then not read
    int* iter;                 // optional device iteration counter k: selects the ping-pong side and the row of diff, and is
                               // incremented by the last CTA (the whole ADMM loop then runs from one captured graph)
    int iter_max;              // with `iter`: the loop condition is cleared after iter_max iterations, on convergence or on an error flag
    int step;                  // without `iter` (host-driven loop): iteration number of this launch -- sequence number and payload
                               //     half of the peer exchange, so that a rank running ahead never reads the previous iteration's slot
    const int* err_a;          // optional error flags (infeasible home, failed QP column): stop the device loop
    const int* err_b;
    unsigned long long cond_loop;   // cudaGraphConditionalHandle of the ADMM while node (use_cond != 0)
    int use_cond;
    double* gamma;             // [Hp][T]  in: G[k]  out: G[k+1]
    double* p_est;             // [Hp][T]  out: P_est[k+1], home-major
    double* z_t;               // [T][Hp]  out: next projection target
    double* g_next;            // optional [T][Hp] (may alias g_t): [z]_+, the next utility iterate of columns without multipliers
    void* gbf_next;            // optional [T][Hp] __nv_bfloat16 copy of g_next
    double* diff_k;            // [Hp]     out: row k of diff (row 0 when `iter` is given; the kernel adds k * Hp)
    ResidualOut* res;
    PeerReduce peer;
    double* partials;          // [2][gridDim.x] per-CTA partial sums: the last CTA adds them in a fixed order (reproducible residuals)
    int Hp, T;
    double kappa, tol, count;  // count = real homes * T
};

cudaError_t launch_dual_update(const DualParams& P, cudaStream_t stream);

// ---- utility_qp.cu
struct QpParams {
    const FeederDev* feeders;
    const double* Rpool;
    const double* rn2;     // [Hp]  squared row norms of the sensitivity blocks
    const double* rmax;    // [Hp]  largest entry of every row of the sensitivity blocks
    int* cand;             // [ncols] set by the screening pass: some row has v~ above the safe threshold
    int* queue;            // work-queue head of the persistent warp kernel (= order_count + kQpLists)
    const double* z_t;     // [T][Hp]
    double* lam_t;         // [T][Hp]   multipliers (dense storage, sparse content)
    double* g_t;           // [T][Hp]   out: projection = P_est[k+1]
    double* v_t;           // [T][Hp]   in (step mode): R g of the stored iterate
    void* gbf_t;           // optional [T][Hp] __nv_bfloat16 copy of g, written with it
    const float* v32_t;    // optional [T][Hp]: BF16-screened voltages; v_t is then filled here (exact for candidates)
    int* wcount;           // [ncols]
    int* widx;             // [ncols][kWMax]
    int* status;           // [ncols] 0 running, 1 converged, 2 working set overflow
    int* inner_ok;         // [ncols] 1: restricted problem solved to tolerance; 2: handed to the next class
                           //         untouched since the last screening pass (picked up by the sweep launch)
    int* n_running;        // columns still running after this launch
    unsigned long long* newton_its;
    int* max_ws;
    unsigned long long* flops;   // algorithmic FP64 flops executed by the QP kernels
    unsigned long long* cols;    // columns that entered a QP kernel
    int* n_failed;         // columns whose working set overflowed kWMax
    int* cls;              // [ncols] instantiation that owns the column (see qp_class_cap)
    int* n_cls;            // [kQpClasses] running columns per class after this round
    const int* order;      // optional [kQpLists][ncols] work lists (order_columns_kernel)
    const int* order_count;   // [kQpLists + 1]
    int4* order4;          // warp-kernel lists [kQpLists - kQpClasses][ncols]: {column, first home, n | ld << 16, R offset / 16}
    int sweep;             // 1: this launch only takes columns handed over during the current round
    int list0, nlists;     // work lists [list0, list0 + nlists) this launch of a warp kernel drains (one queue) ...
    int list_extra;        // ... followed by this list (-1: none)
    int warp_m_max;        // warm working sets above this size start in class 1 (qp_init_kernel)
    int warp_m_max_big;    // the same for zones of more than 128 residences (longer columns)
    int ncols;
    long long* trace;      // optional debug [ncols][12]: start ns, end ns, smid, class/m/pieces, phase cycles ...
    unsigned long long* dbg;  // optional [4 + 5*kQpClasses]: counts, then per-class phase cycles
    int T;
    int64_t Hp;
    double u, tol;
    int init;              // 1: first launch of a utility solve (warm start from lam_t)
    int inner_max;
    int* round_ctr;        // device counter of the working-set rounds of the current utility solve (reset by qp_init_kernel);
                           // order_columns_kernel called with mode < 0 takes its mode from it
    unsigned long long cond_round;   // cudaGraphConditionalHandle of the working-set while node (use_cond != 0)
    int use_cond;
};

// End of a working-set round inside a captured graph: decides whether another round runs.
struct RoundEndParams {
    const int* n_running;
    const int* n_failed;
    const int* infeasible;
    int* round_ctr;
    int* noconv;                 // set when round_max rounds did not finish the solve
    unsigned long long* rounds_total;
    int round_max;
    unsigned long long cond_round;
    int use_cond;
};
cudaError_t launch_round_end(const RoundEndParams& P, cudaStream_t stream);

// Captured loop: IF-node conditions of the CTA classes first_gated.. from their work-list counts.
struct ClassGateParams {
    const int* order_count;
    unsigned long long cond[kQpClasses];
    int first_gated;
};
cudaError_t launch_class_gate(const ClassGateParams& P, cudaStream_t stream);
cudaError_t qp_warp_prepare();       // function attributes of every warp-kernel instantiation on the current device
cudaError_t screen_prepare();
cudaError_t screen_tc5_prepare();

cudaError_t launch_utility_qp(const QpParams& P, int grid, int cls, cudaStream_t stream);
// ---- utility_qp_warp.cu
int qp_warp_max_n();
cudaError_t launch_qp_init(const QpParams& P, int max_warp_n, cudaStream_t stream);
int qp_warp_ctas_per_sm();
int qp_warp_m_max_default();
cudaError_t launch_utility_qp_warp(const QpParams& P, int nj, int ctas_per_sm, cudaStream_t stream);
// one-row columns of the small zones (lists kQpClasses+2, +3): everything in registers, high occupancy;
// columns that turn out to need more are appended to list kListLeftover for the general kernel
cudaError_t launch_utility_qp_fast(const QpParams& P, cudaStream_t stream);
// mode 0: first round of a solve (columns without multipliers and without screening candidates finish here);
// mode 1: later rounds (every running column); mode 2: sweep (columns handed over in this round)
cudaError_t launch_order_columns(const QpParams& P, int mode, int* order, int* order_count, cudaStream_t stream);

// ---- tree_newton.cu: the operator QP of a large radial zone, one CTA per column, all linear algebra on the tree
struct NewtonZone {             // one zone of the Newton path
    int feeder;                 // index of the zone in the solver
    int nn, nlev, n;            // nodes (after the contraction of negligible edges), tree levels, residences
    int wn;                     // max(nn, n): entries per column in the work pools
    int col0;                   // first column of the zone in the launch (columns are zone-major, hour-minor)
    int64_t node_off;           // offset of the zone in the static node pools
    int64_t home_off;           // offset of its node-sorted home list
    int64_t lvl_off;            // offset of its nlev + 1 level offsets
    int64_t ws_off;             // offset (entries) of its T columns in the work pools
    double scale;               // scale of the Hessian shift
};
struct NewtonParams {
    const NewtonZone* zones;
    int n_zones;
    const int* lvl;             // level offsets, breadth-first node numbering
    const int* parent;          // [nodes] parent (breadth-first index), -1: child of the substation
    const int2* child;          // [nodes] {first child, number of children}
    const int2* homes;          // [nodes] {first, number} of the node's residences in the node-sorted home list
    const double* rho;          // [nodes] 2 r of the edge above the node
    const int* hlist;           // [homes] home index inside the zone of every node-sorted position
    const int* hnode;           // [homes] node of every node-sorted position
    double* ws;                 // work pools: kNewtonWsDoubles double arrays of ws_stride entries ...
    double4* ws4;               // ... kNewtonWs4 double4 arrays ...
    double2* ws2;               // ... kNewtonWs2 double2 arrays ...
    int* wsi;                   // ... kNewtonWsInts int arrays
    int64_t ws_stride;
    const FeederDev* feeders;
    const double* z_t;          // [T][Hp]
    double* lam_t;              // [T][Hp]
    double* g_t;                // [T][Hp]
    int* status;                // [ncols]
    int* inner_ok;
    int* wcount;
    int* noconv;                // raised by a column that does not reach the tolerance
    double* dbg_dump;           // optional [8][nn]: x, v, flags, lam, nf, zf, mu, src of one guess of one column (REVS_NEWTON_DUMP=col,outer,guess)
    int dbg_dump_col, dbg_dump_outer, dbg_dump_guess;
    double* dbg_trace;          // optional [columns][16][4]: per outer iteration kkt, solves so far (< 0: guesses cycled), step (< 0: -tau of the safeguard), active rows
    int* dbg_col;               // optional [2 * columns]: tree solves and outer iterations of every column (REVS_DEBUG)
    unsigned long long* newton_its;
    unsigned long long* cols;
    unsigned long long* flops;
    int* max_ws;
    int T;
    int64_t Hp;
    double u, tol;
};
struct NewtonZoneHost {
    std::vector<int> lvl, parent, child0, nchild, home0, nhome, hlist, hnode;
    std::vector<double> rho;
    double scale = 1.0;
};
void newton_build_zone(int n_nodes, const int* parent, const double* r, int n_res, const int* res_node, NewtonZoneHost& Z);
cudaError_t launch_tree_newton(const NewtonParams& P, int n_cols, cudaStream_t stream);
constexpr int kNewtonWsDoubles = 18, kNewtonWs4 = 3, kNewtonWs2 = 2, kNewtonWsInts = 3;

// ---- contract_f64.cu
int contract_tile_rows(int T);
cudaError_t launch_contract(const ContractProblem* d_problems, const ContractTile* d_tiles, int n_tiles,
                            int T, int mode, double v2, cudaStream_t stream);

cudaError_t launch_gather_wait(const unsigned long long* flags, int world, unsigned long long seq, int* timeout, cudaStream_t s);

// ---- screen_bf16.cu
int screen_tile_rows();
cudaError_t launch_to_bf16(const double* in, void* out, size_t n, cudaStream_t s);
cudaError_t launch_screen(const ScreenProblem* d_problems, const ContractTile* d_tiles, int n_tiles, int T, double thr,
                          cudaStream_t stream);

// ---- screen_tc5.cu (tcgen05 / TMEM / TMA implementation of the same contraction)
int screen_tc5_tile_rows();
size_t screen_tc5_map_bytes();
uint32_t screen_tc5_box_rows_a();
uint32_t screen_tc5_box_rows_b();
cudaError_t screen_tc5_encode(void* host_map, const void* gptr, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                              uint32_t box_rows);
cudaError_t launch_screen_tc5(const ScreenProblem* d_problems, const ContractTile* d_tiles, int n_tiles, const void* d_maps_a,
                              const void* d_map_b, const int* d_b_col0, int T, double thr, cudaStream_t stream);

// ---- feeder_build.cu
cudaError_t launch_sens_voltage(const int* parent, const double* cumr, const int* row_node,
                                const int* res_node, int n_rows, int n_res, double* out, int ld,
                                cudaStream_t s);
cudaError_t launch_sens_voltage_batched(const FeederDev* feeders, int n_feeders, int max_n, const int64_t* node_off,
                                        const int* parent, const double* cumr, const int* res_node, double* Rpool,
                                        cudaStream_t s);
cudaError_t launch_sens_flow(const int* parent, const int* row_node, const int* res_node, int n_rows,
                             int n_res, double* out, int ld, cudaStream_t s);
cudaError_t launch_row_norms(const FeederDev* feeders, int n_feeders, const double* Rpool, double* rn2, double* rmax,
                             cudaStream_t s);
cudaError_t launch_pack_rows(const double* src, double* dst, const int64_t* hmap, int64_t H, int w, int to_padded,
                             cudaStream_t s);
cudaError_t launch_hour_mask(const double* p_ev, const int64_t* hmap, int64_t H, int T, unsigned long long* out, cudaStream_t s);
cudaError_t launch_to_time_major(const double* in, int n, int T, double* out, int64_t ld, cudaStream_t s);
// Host: breadth-first numbering of a zone tree (nodes topological, parent -1 = substation), the layout of the
// tree-Newton and network-check kernels.  Roots in index order, then level by level the children of every node in
// index order, so the children of a node are contiguous in the next level; the residences of a node are listed by
// ascending home index.
struct BfsTree {
    std::vector<int> order;           // [nodes] position -> node
    std::vector<int> lvl;             // [levels + 1] first position of every level, then the node count
    std::vector<int> parent;          // [nodes] position of the parent, -1: root
    std::vector<int> child0, nchild;  // [nodes] position of the first child (0 without children), number of children
    std::vector<int> res0, nres;      // [nodes] the node's residences: entries res0.. of res
    std::vector<int> res;             // [residences] home indices grouped by node position
};
void bfs_tree(int n_nodes, const int* parent, int n_res, const int* res_node, BfsTree& B);

// ---- network_check.cu
constexpr int kNetMaxSteps = 32;                      // steps per CTA (G) at most
constexpr size_t kNetSmemSmall = 112 * 1024;          // state of a CTA of the first class: two CTAs per SM
constexpr size_t kNetSmemMax = 224 * 1024;            // one step of a zone above this (28,672 nodes) runs on global scratch
struct NetNode {          // one node of a zone in breadth-first position (children of a node are contiguous in the next level)
    double r;             // resistance of the edge above the node: cumr[i] - cumr[parent[i]]
    int node;             // local node index (row of the outputs)
    int parent;           // breadth-first position of the parent, -1 = substation
    int child0, nchild;   // breadth-first positions of the children
    int res0, nres;       // the node's residences: entries res0.. of the zone's residence list (ascending home index)
};
struct NetZone {
    int64_t node0, lvl0, res0;    // first entry of the zone in the node / level / residence pools
    int64_t home_row;             // padded row of the zone's first home in the [Hp][T] schedule
    int64_t out_row;              // first row of the zone in the [total nodes][T] outputs
    int n_nodes, depth, lg;       // lg: log2 of the steps per CTA
    int n_res;                    // residences
};
struct NetCta { int zone, t0; int64_t gstate; };     // gstate: offset of the state in the global scratch, -1: shared memory
struct NetArg { double v; int zone, pad_; int64_t loc; };   // a maximum and where: loc = index * T + step
struct NetPartial { NetArg drop, exc, load; unsigned long long rows, low, over; };
struct NetParams {
    const NetZone* zones;
    const NetNode* nodes;
    const int* levels;            // per zone: depth + 1 breadth-first positions
    const int* res;               // per zone: local home indices, grouped by node
    const NetCta* ctas;
    const double* P;              // [Hp][T]
    const double* scale;          // [total nodes] or null (= 1)
    double* voltage;              // [total nodes][T] or null
    double* loading;              // [total nodes][T] or null
    double* drop;                 // [Hp * T] or null: D at every residence, the zone's block [T][n_res] at home_row * T
    double* gstate;               // global scratch of the zones above kNetSmemMax
    NetPartial* part;             // [CTAs]
    int T;
    double v2, u, low, row_tol;   // vset^2, vhigh^2 - vset^2, vset^2 - vlow^2, tolerance of the row count
};
// R[i,h] of two residences on the breadth-first positions a, b of their nodes: 2 cumr at the lowest common ancestor
// (0 when they hang on different roots).  A larger position is never above a smaller one, so moving the larger one up
// never passes the ancestor.
__device__ __forceinline__ double lca_r(const NetNode* __restrict__ nd, const double* __restrict__ cumr, int a, int b) {
    while (a != b) {
        if (a > b) a = nd[a].parent;
        else b = nd[b].parent;
        if (a < 0 || b < 0) return 0.0;
    }
    return 2.0 * cumr[nd[a].node];
}
struct NetHost {                  // host side of the arrays above, built once per set of trees
    std::vector<NetZone> zones;
    std::vector<NetNode> nodes;
    std::vector<int> levels, res, lists, zone_cta;
    std::vector<NetCta> ctas;
    int class_off[4] = {0, 0, 0, 0};        // lists[class_off[c] ..] = CTAs of class c: shared <= kNetSmemSmall, shared, global
    size_t class_smem[3] = {0, 0, 0};
    int64_t gstate_doubles = 0, total_nodes = 0;
};
void net_add_zone(NetHost& h, int n_nodes, const int* parent, const double* cumr, int n_res, const int* res_node,
                  int64_t home_row);
void net_finish(NetHost& h, int T);
// log2 of the steps per CTA of a zone whose state is `one` bytes per step, and the class of its CTAs (NetHost::class_off)
int net_zone_lg(size_t one, int T, int* cls);
cudaError_t launch_network_check(const NetParams& P, const int* d_list, int n_ctas, size_t smem, cudaStream_t s);
cudaError_t launch_network_reduce(const NetPartial* part, const int* zone_cta, int n_zones, double* zone_worst,
                                  NetPartial* out, cudaStream_t s);

// ---- repair.cu: greedy voltage repair of the schedule, one CTA per zone
constexpr int kRepairSmemMaxN = 2048;   // zones above this many residences keep their state in the global scratch
constexpr int kRepairMaxT = 256;        // longest horizon (home_solve.cu)
struct RepairParams {
    const NetZone* zones;         // the network check's breadth-first arrays
    const NetNode* nodes;
    const int* res;
    const double* cumr;           // [total nodes] cumulative resistance of every node, zone z at zones[z].out_row
    const double* zone_worst;     // [zones][3] of the network check of the schedule: zones with excess > row_tol run
    const double* load;           // [Hp][T]
    const double* rating;         // [Hp]
    const double* cost;           // [T]
    const int *start, *end, *n_min;   // [Hp]
    double* D;                    // [Hp * T] drops of the schedule at the residences (NetParams::drop), updated
    double* P;                    // [Hp][T] in: the schedule, out: the repaired schedule
    double* p_ev;                 // [Hp][T] in: the charger power, out: the repaired one
    char* gws;                    // global scratch of the zones above kRepairSmemMaxN ...
    const int64_t* ws_off;        // ... [zones] byte offset of the zone's state in it, -1: shared memory
    int32_t* info;                // [zones][3] status, moves, drops
    int T;
    double u, row_tol;
};
size_t repair_ws_bytes(int n_res, int T);     // bytes of a zone's state
cudaError_t launch_repair(const RepairParams& P, int n_zones, size_t smem, cudaStream_t s);

// ---- central.cu: bracket of the centralized optimum per zone (priced selections, Lagrangian ascent, two repairs)
struct CenSelectParams {          // one warp per home: e*(y), or the most expensive SOC-feasible hours
    const NetZone* zones;
    const int* hzone;             // [Hp] zone of every home, -1: padding (EV homes only are read)
    const double* ry;             // zone blocks [T][n]: R y at the residences (NetParams::drop), or null (y = 0)
    const double *load, *rating, *cost;
    const uint8_t* has_ev;
    const int *start, *end, *n_min, *n_max;
    double* P;                    // [Hp][T] out: load + rating e
    double* p_ev;                 // [Hp][T] out: rating e
    int* infeasible;              // set when a home's n_min exceeds its window or n_max
    int64_t Hp;
    int T;
    int most_expensive;           // 1: reduced cost -rating c (ry ignored)
};
struct CenZone { double lb, ub, theta; int stall, done, steps, pad_; };
struct CenAscentParams {
    const NetZone* zones;
    const double* cost;           // [T]
    const double* P;              // [Hp][T] e*(y) of this evaluation
    const double* D;              // zone blocks [T][n]: R P
    double *y, *ybest;            // [Hp][T]
    const double *cost1, *cmax;   // [zones] cost of the repaired e*(0), C_max
    const int32_t* info1;         // [zones][3] repair of e*(0)
    CenZone* state;               // [zones]
    int k, iters, T;
    double u;
};
struct CenFinalParams {
    const NetZone* zones;
    const CenZone* state;
    const double *cost1, *cost2, *cmax;
    const int32_t *info1, *info2;
    double *P1, *p_ev1;           // [Hp][T] repaired e*(0); out: the kept schedule
    const double *P2, *p_ev2;     // [Hp][T] repaired e*(y_best)
    double* bounds;               // [zones][2] LB, UB
    int32_t* info;                // [zones][3] status, ascent steps, moves + drops of the kept start
    int T;
};
cudaError_t launch_central_select(const CenSelectParams& P, cudaStream_t s);
cudaError_t launch_central_ascent(const CenAscentParams& P, int n_zones, cudaStream_t s);
cudaError_t launch_central_cost(const NetZone* zones, int n_zones, const double* cost, const double* P, int T,
                                double* out, cudaStream_t s);
cudaError_t launch_central_final(const CenFinalParams& P, int n_zones, cudaStream_t s);

// ---- certify.cu: certificate of voltage infeasibility per zone (base load, counting over the top-K homes of a row)
constexpr int kCertTopK = 32;     // homes of largest coefficient per residence row that the counting rule looks at
struct CertParams {
    const NetZone* zones;         // the network check's breadth-first arrays
    const NetNode* nodes;
    const int* res;
    const double* cumr;           // [total nodes], zone z at zones[z].out_row
    const int* hzone;             // [Hp] zone of every padded home row, -1: padding
    const double* D;              // zone blocks [T][n]: R load at the residences (NetParams::drop)
    const double* rating;
    const uint8_t* has_ev;
    const int *start, *end, *n_min, *n_max;
    int* hpos;                    // [Hp] out: breadth-first position of every residence's node
    unsigned long long* key;      // [zones] packed witness of kind 2 (atomicMax)
    int32_t* cert;                // [zones][4] out: kind, residence, k or step, need - cap
    int* flag;                    // out: |1 a home's n_min exceeds its window or n_max, |2 a non-finite or negative rating
    int64_t Hp;
    int T;
    double u, thr;                // vhigh^2 - vset^2, row_tol + 1e-12
};
cudaError_t launch_certify(const CertParams& P, int n_zones, cudaStream_t s);

// ---- hosting.cu: hosting capacity of a schedule, per residence and step and per zone and step
struct HcCta { int zone, t0, lg, pad_; int64_t gstate; };  // lg: log2 of the steps; gstate: global scratch offset, -1: shared
struct HcParams {
    const NetZone* zones;         // the network check's breadth-first arrays
    const NetNode* nodes;
    const int* levels;
    const int* res;
    const HcCta* ctas;
    const double* cumr;           // [total nodes], zone z at zones[z].out_row
    const double2* wn;            // [nodes pool] per breadth-first position: {W, N}, the drop and flow of 1 kW everywhere
    const double* P;              // [Hp][T]
    const double* scale;          // [total nodes] signed 1/rating per edge (0 = unrated), or null: no edge is rated
    const uint8_t* has_ev;        // [Hp]
    const double* rating;
    const int *start, *end;
    double* cap;                  // [Hp][T] out, or null
    double* uniform;              // [zones][T] out, or null
    double* gstate;               // global scratch of the zones above kNetSmemMax (two doubles per node)
    unsigned long long* part;     // [CTAs][3] window steps, open window steps, thermally bound pairs
    int T;
    double ur;                    // u + row_tol
};
struct HcHost {                   // host side of the hosting CTAs, built once per set of trees
    std::vector<HcCta> ctas;
    std::vector<int> lists, zone_cta;
    std::vector<double2> wn;
    int class_off[4] = {0, 0, 0, 0};
    size_t class_smem[3] = {0, 0, 0};        // dynamic shared memory of each class, at least the final reduction's
    int64_t gstate_doubles = 0;
};
void hc_prepare(const NetHost& h, int T, HcHost& out);
cudaError_t launch_hosting(const HcParams& P, const int* d_list, int n_ctas, size_t smem, cudaStream_t s);
cudaError_t launch_hosting_reduce(const unsigned long long* part, const int* zone_cta, int n_zones, int64_t* counts,
                                  cudaStream_t s);

}  // namespace revs
