/*
 * revs_admm.h -- C ABI of the B200-native REVS distributed EV-charging ADMM path.
 *
 * Drop-in boundary: these are the entry points a maintainer of the reference
 * (rounak-meyur/revs-admm, pure Python + Gurobi) would bind with ctypes to replace the
 * hot path of lpsolver.py.  Plain pointers and sizes only; every array is dense,
 * row-major, float64 unless stated.  All functions return REVS_OK (0) or an error
 * code; revs_last_error() gives the text.  There is NO CPU fallback: every entry point
 * fails with REVS_ERR_CUDA when no sm_100 device is usable.
 *
 * Reference interface replaced by each entry point (file:line in /root/reference):
 *
 *   revs_set_sensitivity / revs_set_feeder_tree(s) lpsolver.py:17-26  compute_Rmat()
 *                                                 lpsolver.py:183-194 Utility.network()
 *   revs_set_homes / revs_set_tariff              lpsolver.py:45-58   Home.__init__ inputs
 *                                                 extract.py:91-132   get_homes_ev_param()
 *   revs_solve_admm                               lpsolver.py:242-290 solve_ADMM()
 *   revs_admm_begin / revs_admm_step              lpsolver.py:254-287 one while-iteration
 *   revs_home_step                                lpsolver.py:44-160  Home(...).solve()
 *   revs_utility_step                             lpsolver.py:163-238 Utility(...).solve()
 *   revs_solve_individual                         lpsolver.py:430-460 solve_residence()
 *   revs_reliability                              drawing.py:29-78    compute_flows(),
 *                                                                     compute_voltage()
 *   revs_network_check                            drawing.py:29-78    the same for every zone at once
 *   revs_repair_schedule                          no reference counterpart (a voltage-feasible binary schedule)
 *   revs_central_bracket                          lpsolver.py:463-502 solve_central(), bracketed per zone
 *   revs_certify_infeasible                       lpsolver.py:463-502 solve_central(), zones proved infeasible
 *   revs_hosting_capacity                         no reference counterpart (the extra load every home can take)
 *   revs_get_results / revs_get_schedule(_ld)     lpsolver.py:289-290 return diff,P_sch,S,C
 *   revs_set_option / revs_get_stats / revs_version / revs_last_error / revs_device_count /
 *   revs_reliability_sharded / revs_gather_export / revs_gather_attach
 *                                                 drawing.py:29-78 for one feeder over several GPUs (rows partitioned)
 *   revs_comm_export / revs_comm_attach / revs_comm_detach
 *                                                 no reference counterpart (library plumbing; the reference is one process)
 */
#ifndef REVS_ADMM_H
#define REVS_ADMM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define REVS_OK 0
#define REVS_ERR_ARG 1          /* bad argument / call order                          */
#define REVS_ERR_CUDA 2         /* CUDA error or no usable device                     */
#define REVS_ERR_INFEASIBLE 3   /* a home sub-problem has no solution (lpsolver.py:154)*/
#define REVS_ERR_NOCONV 4       /* utility QP hit its iteration / working-set limit    */

#define REVS_REL_VOLTAGE 0      /* out = sqrt(vset^2 - S_v P)   (drawing.py:75)        */
#define REVS_REL_FLOW 1         /* out = scale[row] * (S_f P)   (drawing.py:56-58)     */
#define REVS_REL_DROP 2         /* out = S_v P                  (R@P of lpsolver.py:192)*/

typedef struct revs_solver revs_solver;

/* counters of the last revs_solve_* call (what ran on the device) */
typedef struct revs_stats {
    int64_t kernel_launches;      /* kernels of this library launched                  */
    int64_t gemm_launches;        /* ... of which sensitivity contractions             */
    int64_t gemm_full_launches;   /* ... of which over all columns (first round of an iteration) */
    int64_t qp_outer_iterations;  /* utility working-set rounds, summed over ADMM iters */
    int64_t qp_newton_iterations; /* restricted Newton steps, summed over columns       */
    int32_t admm_iterations;
    int32_t max_working_set;      /* largest per-(feeder,hour) working set seen         */
    double primal_residual;       /* ||P_est-P_sch||_F / sqrt(H T), last iteration      */
    double dual_residual;         /* kappa ||P_sch-P_sch_prev||_F / sqrt(H T)           */
    double qp_flops;              /* algorithmic FP64 flops of the utility QP kernels   */
    float gemm_ms;                /* device time in sensitivity contractions (events)   */
    float gemm_full_ms;           /* ... of which the launches over ALL (feeder,hour) columns */
    float home_ms;                /* device time in the batched home solve              */
    float dual_ms;                /* device time in the fused dual/residual kernel      */
    float qp_ms;                  /* device time in the per-column QP kernels (both)    */
    float qp_big_ms;              /* ... of which the |W|>32 instantiation              */
    float total_ms;               /* device time of the whole solve                     */
    float qp_warp_ms;             /* ... of qp_ms: warp-per-column kernels (zones <= 256) */
    float qp_init_ms;             /* ... of qp_ms: start-of-solve kernel                 */
    int64_t qp_columns;           /* (zone,hour) columns that entered a QP kernel, summed over rounds */
    int64_t qp_warp_rounds;       /* working-set rounds in which the warp-per-column kernels ran */
} revs_stats;

const char* revs_last_error(void);
int revs_version(void);
int revs_device_count(int* count);

/* A solver owns the device state of a batch of feeders that live on ONE GPU.
 * feeder_off[n_feeders+1]: residences of feeder f are homes feeder_off[f]..feeder_off[f+1]-1
 * of every [H, *] array below (H = feeder_off[n_feeders]).  T = horizon length. */
int revs_create(revs_solver** out, int device, int n_feeders, const int64_t* feeder_off, int T);
int revs_destroy(revs_solver* s);

/* Residence-by-residence voltage sensitivity block R_res (n_f x n_f, symmetric, >=0)
 * of one feeder, from host memory. */
int revs_set_sensitivity(revs_solver* s, int feeder, const double* R_res);

/* Same block built ON THE DEVICE from the radial feeder itself: n_nodes non-substation
 * nodes in topological order (parent[i] < i, -1 = substation), r[i] = resistance of the
 * edge above node i, res_node[n_f] = node index of each residence.  Also enables
 * revs_reliability() on arbitrary nodes / edges of this feeder. */
int revs_set_feeder_tree(revs_solver* s, int feeder, int n_nodes, const int32_t* parent,
                         const double* r, const int32_t* res_node);

/* All feeders of the solver at once (one upload, one kernel): node_off[n_feeders+1] offsets
 * into the concatenated parent / r arrays (parent indices are local to their feeder),
 * res_node [H] in the home order of revs_create (node indices local to the feeder). */
int revs_set_feeder_trees(revs_solver* s, const int64_t* node_off, const int32_t* parent,
                          const double* r, const int32_t* res_node);

/* Per-home inputs (host).  load [H,T] kW; has_ev [H]; rating kW, capacity kWh, initial
 * SOC, start/end = plug-in window [start,end) in steps.  EV arrays are ignored where
 * has_ev==0. */
int revs_set_homes(revs_solver* s, const double* load, const uint8_t* has_ev,
                   const double* rating, const double* capacity, const double* initial,
                   const int32_t* start, const int32_t* end);
int revs_set_tariff(revs_solver* s, const double* cost /* [T] */);

/* Full ADMM run == solve_ADMM(): iter_max iterations from P_est=P_sch=Gamma=0.
 * tol<=0 reproduces the reference (always iter_max iterations); tol>0 stops early when
 * both residuals of revs_stats fall below tol.  iters_done may be NULL. */
int revs_solve_admm(revs_solver* s, double kappa, int iter_max, double vset, double vlow,
                    double vhigh, double tol, int* iters_done);

/* The same loop one iteration at a time (multi-GPU drivers all-reduce the residual
 * sums between steps).  sums[3] = {sum (P_est-P_sch)^2, sum (P_sch-P_sch_prev)^2, H*T}
 * over this solver's homes. */
int revs_admm_begin(revs_solver* s, double kappa, int iter_max, double vset, double vlow,
                    double vhigh);
int revs_admm_step(revs_solver* s, double sums[3]);

/* The two sub-problems on their own, host in/out, all homes of the solver at once.
 * revs_home_step  == Home(cost, homedata, p_est, p_sch, gamma, kappa).solve() per home:
 *   P_sch_new = g_opt [H,T], P_ev = p_opt [H,T] (either may be NULL).
 * revs_utility_step == Utility(graph, P_est, P_sch, Gamma, kappa, vset, vlow, vhigh).solve():
 *   P_est_new = g_opt [H,T]; lam0 (may be NULL) warm-starts the voltage-row multipliers,
 *   lam_out (may be NULL) returns them, both [H,T]. */
int revs_home_step(revs_solver* s, double kappa, const double* p_est, const double* p_sch,
                   const double* gamma, double* P_sch_new, double* P_ev);
int revs_utility_step(revs_solver* s, double kappa, double vset, double vlow, double vhigh,
                      const double* p_est, const double* p_sch, const double* gamma,
                      const double* lam0, double* P_est_new, double* lam_out);

/* Results of the last ADMM run, to host.  Any pointer may be NULL.
 * P_sch [H,T], P_ev [H,T], SOC [H,T+1], diff [diff_rows,H] (lpsolver.py:284): one row per iteration
 * that ran; REVS_ERR_ARG when diff_rows is smaller than that (nothing is written past the buffer). */
int revs_get_results(const revs_solver* s, double* P_sch, double* P_ev, double* SOC,
                     double* diff, int diff_rows);
/* The same results in compact form: the schedule P_sch [H,T] and the charging decisions as bit masks,
 * hour_mask [H, mask_words] with mask_words = ceil(T/64), bit (t % 64) of word t/64 set when the charger of the
 * home runs in step t.  S = rating * bit and the SOC recursion C (lpsolver.py:105-108) follow from the mask and
 * the per-home inputs the caller already holds, so a third of the bytes of revs_get_results cross PCIe. */
int revs_get_schedule(const revs_solver* s, double* P_sch, uint64_t* hour_mask, int mask_words,
                      double* diff, int diff_rows);
/* revs_get_schedule with a row stride for diff: row k of the convergence values goes to diff + k * diff_ld
 * (diff_ld >= H, in doubles), so that several solvers sharing one GPU write their column blocks of one
 * [iterations, all homes] array (lpsolver.py:284 keeps one such array) straight from the device, without a host copy. */
int revs_get_schedule_ld(const revs_solver* s, double* P_sch, uint64_t* hour_mask, int mask_words,
                         double* diff, int diff_rows, int64_t diff_ld);

/* Utility-side iterates of the last run: P_est [H,T], Gamma [H,T]. */
int revs_get_estimate(const revs_solver* s, double* P_est, double* Gamma);

/* Individual optimum of every home == solve_residence() per home. */
int revs_solve_individual(revs_solver* s, double* P_res, double* P_ev, double* SOC);

/* LinDistFlow reliability check of a schedule on one feeder (needs set_feeder_tree):
 * rows = node indices (voltage/drop) or edge indices (= child-node index of the edge,
 * flow).  P [n_f,T] host schedule of the feeder's residences, or NULL to use the last
 * ADMM result.  out [n_rows,T] host.  scale [n_rows] only for REVS_REL_FLOW (signed
 * 1/rating), may be NULL (=1). */
int revs_reliability(revs_solver* s, int feeder, int kind, int n_rows, const int32_t* rows,
                     const double* scale, double vset, const double* P, double* out);

/* Network check of the whole population (drawing.py:29-78 for every zone of the solver at once): the voltage at
 * every node and the flow on every line, per step, and where the limits are violated.  One kernel walks every zone's
 * tree (leaves -> root: flows F, root -> leaves: squared-voltage drops D = R P), O(nodes x T), no sensitivity
 * matrix; every zone needs its tree (revs_set_feeder_tree(s)).
 * source: REVS_NET_SCHEDULE / REVS_NET_ESTIMATE (schedule / operator estimate of the last ADMM run, already on the
 * device, P ignored), REVS_NET_HOST (P [H,T] from the host, compact home order of revs_create), REVS_NET_REPAIRED
 * (the repaired schedule of revs_repair_schedule, below) or REVS_NET_CENTRAL (the kept schedule of
 * revs_central_bracket, below).
 * "Total nodes" are the nodes of all zones concatenated in zone order (node_off of revs_set_feeder_trees); rows of
 * voltage / loading, and scale, follow it.  voltage = sqrt(vset^2 - D) (REVS_REL_VOLTAGE), loading = scale * F
 * (REVS_REL_FLOW, scale = signed 1/rating per edge, NULL = 1).  voltage, loading, zone_worst and summary may be NULL.
 * Ties of every maximum go to the lowest (zone, node or residence, step); counts are exact: two calls give the same
 * bytes, and the result of a zone does not depend on the other zones of the solver.
 * REVS_ERR_ARG: a zone without tree (the message names it), SCHEDULE / ESTIMATE before any ADMM iteration, HOST
 * without P, REPAIRED before a repair of the current ADMM run, CENTRAL before a bracket of the current homes, tariff and
 * trees, an unknown source, or not vlow <= vset < vhigh.  Synchronous on the utility stream; adds its launches to
 * revs_stats.kernel_launches and changes no other state.  The breadth-first arrays it needs are built on its first
 * call after the trees are set, its scratch on first use; both are kept until revs_destroy. */
#define REVS_NET_SCHEDULE 0   /* P_sch of the last ADMM run (what revs_get_results returns)      */
#define REVS_NET_ESTIMATE 1   /* P_est of the last ADMM run (what revs_get_estimate returns)     */
#define REVS_NET_HOST 2       /* P [H,T] from the host, compact home order of revs_create        */

typedef struct revs_network_summary {
    double drop_max;           /* max over all nodes and steps of (R P) at the node, pu^2 (REVS_REL_DROP)          */
    double v_min;              /* sqrt(vset^2 - drop_max), the REVS_REL_VOLTAGE formula                           */
    int32_t drop_zone, drop_node, drop_step;   /* where (node index local to its zone, as in revs_reliability)    */
    int32_t pad0_;
    double row_excess_max;     /* max over RESIDENCES and steps of (R P)_res - (vhigh^2 - vset^2): the voltage row
                                  of the operator QP (revs_admm_begin); > 0 = violated; -inf without residences  */
    int32_t excess_zone, excess_res, excess_step, pad1_;   /* excess_res: home index local to its zone; -1: none  */
    int64_t rows_violated;     /* (residence, step) pairs with excess > row_tol                                   */
    int64_t nodes_below_vlow;  /* (node, step) pairs with drop > vset^2 - vlow^2                                  */
    double loading_max;        /* max over edges and steps of |scale[e] * flow_e| (REVS_REL_FLOW)                 */
    int32_t loading_zone, loading_node, loading_step, pad2_;
    int64_t edges_overloaded;  /* (edge, step) pairs with |loading| > 1; 0 when scale == NULL                      */
} revs_network_summary;

int revs_network_check(revs_solver* s, int source, const double* P, double vset, double vlow, double vhigh,
                       double row_tol,
                       const double* scale,        /* [total nodes] signed 1/rating per edge, or NULL (= 1)     */
                       double* voltage,            /* [total nodes, T] or NULL                                  */
                       double* loading,            /* [total nodes, T] or NULL                                  */
                       double* zone_worst,         /* [n_feeders, 3]: drop_max, row_excess_max, loading_max     */
                       revs_network_summary* summary);

/* Greedy voltage repair of the last ADMM run's charging decisions (see the header comment for the rule).
 * P_out [H,T] (compact home order) and hour_mask [H, mask_words] may be NULL; zone_info [n_feeders, 3] int32 =
 * {status 0/1/2, hours moved, hours dropped}, may be NULL.  The repaired schedule stays on the device for
 * revs_network_check(REVS_NET_REPAIRED) until the next ADMM run.
 *
 * The rule, zone by zone (R is block-diagonal over zones), with D = R P at the residences, u = vhigh^2 - vset^2 and a
 * row (i, t) violated when D[i,t] - u > row_tol:
 *   1. take the worst violated row (i*, t*) of the steps not marked stuck: largest excess, then lowest residence, then
 *      lowest step (the order of revs_network_check); stop when there is none;
 *   2. the candidates are the homes charging at t*, by relief rating_h R[i*,h] descending, ties to the lowest home;
 *   3. the first candidate charging more than n_min hours (the SOC target) drops hour t*; one at n_min moves it to the
 *      cheapest hour of its plug-in window it does not charge at and that stays feasible (ties: earliest hour);
 *   4. when no candidate can drop or move, t* is marked stuck.
 * Charges only leave violated steps and only enter steps that stay feasible: no feasible step becomes violated, no
 * row's excess grows past max(its input excess, row_tol), every home keeps its SOC window and plug-in window, and the
 * loop ends after at most as many drops and moves as there were charges at violated steps.  Homes whose hours did not
 * change keep their P_sch bytes; changed ones get P = load + (charging ? rating : 0).
 * The rule is a heuristic: it does not look for the cheapest feasible schedule.  Zone status: 0 = no violated row,
 * untouched; 1 = repaired, no violated row left; 2 = violated rows left (e.g. the base load alone violates a row).
 * Needs the tree of every zone (revs_set_feeder_tree(s)).  REVS_ERR_ARG: a zone without tree (named), no ADMM
 * iteration, mask_words != ceil(T/64) with hour_mask, not vset < vhigh, row_tol < 0 or NaN.  Synchronous on the
 * utility stream; adds its launches to revs_stats.kernel_launches and changes no other state (P_sch, P_ev, P_est,
 * Gamma, diff stay as they are). */
int revs_repair_schedule(revs_solver* s, double vset, double vhigh, double row_tol,
                         double* P_out, uint64_t* hour_mask, int mask_words, int32_t* zone_info);
#define REVS_NET_REPAIRED 3   /* the schedule of the last revs_repair_schedule of the current ADMM run  */

/* Bracket of the centralized optimum (the reference's solve_central, lpsolver.py:463-502: minimise the tariff cost
 * under the SOC and voltage rows), zone by zone on the device: UB_z, the cost of a voltage-feasible binary schedule
 * that keeps every home's SOC window and plug-in window, and LB_z, a lower bound on the cost of every such schedule.
 * Needs the homes, the tariff and the tree of every zone; an ADMM run is not needed, and nothing of one is read or
 * changed.  P_out [H,T] (compact home order), hour_mask [H, mask_words], zone_bounds [n_feeders, 2] {LB, UB} and
 * zone_info [n_feeders, 3] int32 {status, ascent steps run, hours moved + dropped by the repair of the kept start}
 * may each be NULL.  The kept schedule stays on the device for revs_network_check(REVS_NET_CENTRAL) until the homes,
 * tariff or trees change.
 *
 * The method, with u = vhigh^2 - vset^2, c the tariff, P = load + rating e (e binary inside the plug-in window,
 * n_min <= sum e <= n_max as in the home solve), R the residences' sensitivity block and y >= 0 one price per
 * (residence, step):
 *   1. priced selection e*(y): every home takes the n_min window hours of smallest reduced cost rating (c_t + (R y)_t),
 *      then further hours while the reduced cost is negative, up to n_max; ties to the earliest hour, exact values;
 *   2. phi(y) = sum c P(y) + sum y (R P(y) - u) is a lower bound on every feasible schedule's cost, at every y;
 *   3. start y = 0 (phi(0) = cost of every home's cheapest SOC-feasible hours); the greedy rule of
 *      revs_repair_schedule applied to e*(0) gives UB_z (+inf when it leaves a violated row);
 *   4. evaluations k = 0..iters of phi(y_k); LB_z = the best; theta_z (from 1) halves after 20 evaluations without a
 *      new best; y <- max(y + theta_z (target_z - phi_z) / ||g_z||^2 (R P - u), 0), g the projected subgradient,
 *      target_z = UB_z when a feasible schedule is known, else C_max_z + 0.01 |C_max_z|.  C_max_z is the cost of the
 *      most expensive SOC-feasible schedule (the n_min dearest window hours, then further hours while c_t > 0, up to
 *      n_max).  A zone stops when UB_z - LB_z <= 1e-9 |UB_z|, g_z = 0, or (without a feasible schedule) LB_z > C_max_z;
 *   5. the greedy repair of e*(y_best) is a second start; the cheaper repaired schedule is kept, ties to the first.
 * Status: 0 = e*(0) meets every row (optimal, LB = UB); 1 = bracketed, LB <= optimum <= UB; 2 = no feasible schedule
 * found (UB = +inf; the kept schedule violates rows); 3 = certified infeasible, LB_z > C_max_z (UB = +inf).
 * Sums run in a fixed order: two calls give the same bytes, and a zone's result does not depend on the other zones.
 * REVS_ERR_INFEASIBLE: a home whose n_min exceeds its plug-in window.  REVS_ERR_ARG: homes or tariff not set, a zone
 * without tree (named), iters < 0, mask_words != ceil(T/64) with hour_mask, not vset < vhigh, row_tol < 0 or NaN.
 * Synchronous on the utility stream; adds its launches to revs_stats.kernel_launches. */
int revs_central_bracket(revs_solver* s, double vset, double vhigh, double row_tol, int iters, double* P_out,
                         uint64_t* hour_mask, int mask_words, double* zone_bounds, int32_t* zone_info);
#define REVS_NET_CENTRAL 4    /* the kept schedule of the last revs_central_bracket                    */

/* Certificate of voltage infeasibility, zone by zone on the device: a proof that no binary schedule keeps every home's
 * SOC window (n_min charging hours at least) and plug-in window and the voltage rows (R P)_i,t - u <= row_tol, or "no
 * proof found".  It covers the zones the Lagrangian bound of revs_central_bracket cannot: that bound equals the LP
 * relaxation's, and a zone whose LP relaxation meets the rows can still have no binary schedule, because a home draws
 * its full rating in every hour it charges.  Needs the homes and the tree of every zone; no tariff or ADMM run.
 *
 * The rule, with u = vhigh^2 - vset^2, D0 = R load at the residences (the network check's drops of the base load),
 * a_h(i) = rating_h R[i,h] (R[i,h] = 2 cumr at the lowest common ancestor of the two residences' nodes), the homes
 * that count = the EV homes with n_min > 0, and a set of charges fitting row (i,t) when (D0[i,t] + s) - u <=
 * row_tol + 1e-12, s the sum of their coefficients (round-to-nearest; the 1e-12 pu^2 margin resolves every rounding
 * in favour of "fits", so no certificate comes from rounding):
 *   kind 1: some row has D0[i,t] - u > row_tol + 1e-12 (the base load alone violates it); witness: the worst such row,
 *           ties to the lowest residence, then the lowest step;
 *   kind 2: for a residence i, S_k = the k homes of largest a_h(i) (ties to the lowest home), k = 1..K,
 *           K = min(32, homes that count); m_t(k) = the largest j such that the j smallest coefficients of the members
 *           of S_k whose window contains t fit row (i,t), added in ascending order; cap_k = sum_t m_t(k),
 *           need_k = sum of n_min over S_k.  cap_k < need_k proves the zone infeasible (R >= 0 and rating >= 0: charges
 *           outside S_k and at other rows only use up slack).  Witness: the (i, k) of the largest need_k - cap_k, ties
 *           to the lowest residence, then the lowest k.
 * A zone of kind 1 reports kind 1.  zone_cert [n_feeders, 4] int32 {kind 0 (no proof) / 1 / 2, residence (local index
 * in the zone, -1 for kind 0), step (kind 1) or k (kind 2) (-1 for kind 0), need_k - cap_k (kind 2, else 0)} and
 * n_certified (zones of kind 1 or 2) may each be NULL.  Every reduction is an integer or total-order maximum: two calls
 * give the same bytes, and a zone's result does not depend on the other zones.
 * REVS_ERR_ARG: homes not set, a zone without tree (named), not vset < vhigh, row_tol < 0 or NaN, an EV home with a
 * negative or non-finite rating.  REVS_ERR_INFEASIBLE: a home whose n_min exceeds its plug-in window (or n_max), as in
 * revs_central_bracket.  Synchronous on the utility stream; adds its launches to revs_stats.kernel_launches and
 * changes no other state (the schedules of revs_repair_schedule and revs_central_bracket stay checkable). */
int revs_certify_infeasible(revs_solver* s, double vset, double vhigh, double row_tol, int32_t* zone_cert,
                            int* n_certified);

/* Hosting capacity of a schedule, zone by zone on the device: for every residence and step, how many more kW its home
 * can draw, with everything else unchanged, before a voltage row or a rated line binds; for every zone and step, how
 * many more kW every residence of the zone can draw at once.  Needs the tree of every zone; no homes, tariff or ADMM
 * run (the counts below read the homes' windows and ratings when they are set, else they are 0).
 *
 * Per zone and step, with u = vhigh^2 - vset^2 and D = R P at the nodes (as in revs_network_check), the residence rows
 * (R P)_i - u <= row_tol of the repair, bracket and certificate, d_a = 2 cumr[a] (R[i,h] = d at the lowest common
 * ancestor of the two residences' nodes), F_a the flow on the edge above node a and s_a the caller's signed 1/rating of
 * that edge (s_a = 0 or scale = NULL: unrated):
 *   sigma_i = (u + row_tol) - D_i, the slack of residence i (u + row_tol formed once, then the subtraction);
 *   home_cap[h,t] = max(0, min(V_h, L_h)), +inf when nothing limits, where
 *     V_h = min over the ancestors a of h's node (the node included) with d_a > 0 of M_a / d_a, M_a = min sigma_i over
 *           the residences below a, and
 *     L_h = min over the rated edges a on h's path of (1 - |s_a| F_a) / |s_a|.
 *   V_h equals min_i sigma_i / R[i,h] over R[i,h] > 0 bit for bit: a correctly rounded division is monotone in both
 *   operands and min sigma / d = min (sigma / d); an ancestor above the true lowest common ancestor has a smaller d, so
 *   its term is never the smaller one while sigma >= 0; a negative slack makes both forms negative, and both clamp to 0.
 *   L_h is exact while no edge is overloaded against its flow (adding load at h raises F on every edge of h's path).
 *   zone_uniform[z,t] = max(0, min(min_i sigma_i / W_i over W_i > 0, min over rated edges a with N_a > 0 of
 *     (1 - |s_a| F_a) / (|s_a| N_a))), W = R 1 the drop of 1 kW at every residence (the network check's recurrences on
 *     P = 1), N_a the residences below edge a: the extra load every residence of the zone can draw at once.
 *   zone_counts[z] = {window_steps: (EV home, step of its plug-in window) pairs; window_steps_open: of those, the pairs
 *     with home_cap >= rating (one more charger fits with nothing else changed); thermal_bound: (home, step) pairs with
 *     L_h < V_h, 0 without scale} (int64).
 * The lower voltage limit vlow is not a row here, nor are non-residence nodes.  home_cap [H,T] (compact home order),
 * zone_uniform [n_feeders, T] and zone_counts [n_feeders, 3] may each be NULL; scale [total nodes] as in
 * revs_network_check.  Every output is a minimum or an integer count: two calls give the same bytes, and a zone's
 * result does not depend on the other zones.
 * source: the five REVS_NET_* sources, with the preconditions of revs_network_check.  REVS_ERR_ARG: those of the
 * source, a zone without tree (named), not vset < vhigh, row_tol < 0 or NaN, a non-finite scale entry.  Synchronous on
 * the utility stream; adds its launches to revs_stats.kernel_launches and changes no other state (the schedules of
 * revs_repair_schedule and revs_central_bracket stay checkable). */
int revs_hosting_capacity(revs_solver* s, int source, const double* P, double vset, double vhigh, double row_tol,
                          const double* scale, double* home_cap, double* zone_uniform, int64_t* zone_counts);

/* The same check with the ROWS PARTITIONED over the GPUs of one box (one process per GPU, every process holds the
 * feeder's tree; BASELINE north_star: "the sensitivity contraction is row-partitioned"): every rank builds and
 * contracts only its block of the requested rows, and the epilogue of the contraction kernel stores each output
 * element straight into the gather buffer of EVERY rank through peer-mapped (NVLink) memory -- the all-gather is
 * fused into the FP64 tensor-core kernel, there is no NCCL call and no extra copy; arrival flags (system-scope
 * release / acquire) close the exchange.  All ranks call it with the same arguments; P (the feeder's whole
 * schedule, [n_f,T]) is required; out [n_rows,T] is complete on every rank.
 * Protocol: revs_gather_export (allocates this rank's buffer for up to capacity_doubles = n_rows*T outputs, returns
 * its 64-byte CUDA IPC handle), exchange the handles on the host, revs_gather_attach with all `world` handles in
 * rank order (<= 16 ranks), a host barrier, then any number of revs_reliability_sharded calls (collective).
 * Replaces drawing.py:29-78 for a feeder too large for one GPU's share of the time; the reference is one process. */
int revs_gather_export(revs_solver* s, int64_t capacity_doubles, void* handle64);
int revs_gather_attach(revs_solver* s, int world, int rank, const void* handles);
int revs_reliability_sharded(revs_solver* s, int feeder, int kind, int n_rows, const int32_t* rows,
                             const double* scale, double vset, const double* P, double* out);

/* Plain sensitivity contraction C[M,T] = A[M,K] @ B[K,T] on the tensor cores (FP64
 * DMMA), host in/out -- exposed so that the GEMM kernel can be tested on its own. */
int revs_contract(int device, int M, int K, int T, const double* A, const double* B, double* C);

/* The in-loop screening contraction on its own: C ~ A @ B with BF16 operands and FP32
 * accumulation (relative error <= 0.5 % for non-negative data).  impl 0 = mma.sync kernel,
 * impl 1 = tcgen05 / TMEM / TMA kernel (T <= 96). */
int revs_screen_contract(int device, int M, int K, int T, const double* A, const double* B, double* C,
                         int impl);

/* Global stopping rule over the GPUs of one box (one process per GPU, each with its own revs_solver over its
 * share of the feeders): the residual sums of revs_stats / revs_admm_step / the tol test of revs_solve_admm then
 * run over ALL ranks.  The all-reduce happens inside the fused dual-update kernel, through mailboxes in peer
 * (NVLink) memory -- no NCCL call, no extra launch, nothing returns to the host.  Protocol: every rank calls
 * revs_comm_export (a 64-byte CUDA IPC handle of its mailbox), the host exchanges the handles (e.g.
 * torch.distributed.all_gather), every rank calls revs_comm_attach with all `world` handles in rank order
 * (<= 16 ranks).  The mailbox is zeroed by attach: synchronise the ranks (a barrier) between attach and the
 * first revs_admm_begin.  All ranks must then make the same sequence of revs_admm_begin / step / solve calls.
 * No reference counterpart (the reference is a single process). */
int revs_comm_export(revs_solver* s, void* handle64);
int revs_comm_attach(revs_solver* s, int world, int rank, const void* handles);
int revs_comm_detach(revs_solver* s);

/* Options: "graph" (default 1) = revs_solve_admm runs the whole loop from one captured CUDA graph whose loops
 * (ADMM iterations, working-set rounds) are decided on the device; 0 = host-driven loop with CUDA-event spans per
 * kernel family in revs_stats (profiling).  "screen" (default 1) = BF16 tensor-core screening of the voltage rows with exact
 * FP64 recheck of the candidates inside the loop; 0 = FP64 DMMA contraction of every row.
 * "screen_impl" = 0 mma.sync screening kernel, 1 tcgen05/TMEM/TMA screening kernel. */
int revs_set_option(revs_solver* s, const char* name, double value);

int revs_get_stats(const revs_solver* s, revs_stats* out);

#ifdef __cplusplus
}
#endif
#endif /* REVS_ADMM_H */
