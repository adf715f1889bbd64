/*
 * miqp_b200.h -- C ABI of the B200-native MIQP backend (libmiqp_b200.so).
 *
 * This is the drop-in boundary for the solver path of bark-simulator/planner-miqp: what
 * the reference does through IBM CPLEX/OPL behind `CplexWrapper::callCplex`
 * (reference src/cplex_wrapper.cpp:65-249) is done here by hand-written sm_100a CUDA
 * kernels.  Plain pointers and sizes only; no C++ or torch types cross this boundary.
 * There is no CPU fallback: every compute entry point returns MIQP_B200_ERR_CUDA when no
 * CUDA device is usable.
 *
 * Entry point                      replaces (reference file:line)
 * -------------------------------  ------------------------------------------------------
 * MiqpB200Problem                  ModelParameters, src/miqp_planner_data.hpp:99-185, as
 *                                  streamed by ModelInputDataSource::read,
 *                                  src/model_input_data_source.cpp:180-275 (polygons as
 *                                  closed edge lists, :150-178)
 * miqp_b200_layout                 decision_variables.mod:10-53 / RawResults,
 *                                  src/miqp_planner_data.hpp:46-97
 * miqp_b200_assemble               IloOplModel::generate(), src/cplex_wrapper.cpp:98 over
 *                                  the cplexmodel .mod files (row instantiation)
 * miqp_b200_sizes                  collectCplexStatistics, src/cplex_wrapper.cpp:680-690
 * miqp_b200_evaluate               objective_function.mod:7-19 + row feasibility
 * miqp_b200_solve_batch            cplex.solve() + collectRawResults +
 *                                  collectSolutionStatus, src/cplex_wrapper.cpp:158-249,
 *                                  :311-448, :672-678; MIP start :494-639
 * miqp_b200_batch_* (resident)     the same solve with the batch already in HBM
 * miqp_b200_batch_run_streaming    the same run, each plan's result handed to a callback in
 *                                  the round its search ends (one result per cplex.solve()
 *                                  of the reference, instead of one per batch)
 * miqp_b200_set_solution_pool      the solution pool of cplex.solve(); its size is
 *                                  SolutionProperties.NrSolutionPool, collectCplexStatistics,
 *                                  src/cplex_wrapper.cpp:680-690
 * miqp_b200_pool_sizes / _fetch    the pool's members (IloCplex::getSolnPoolNsolns /
 *                                  getValues(sol, i)), best first
 * miqp_b200_pool_export / _merge   (no counterpart) the pool of a plan whose frontier is sharded
 *                                  over GPUs: every rank's pool packed for an all-gather, and
 *                                  the pool of the union of the ranks' leaves built from them
 */
#ifndef MIQP_B200_H
#define MIQP_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  MIQP_B200_OK = 0,
  MIQP_B200_ERR_CUDA = -1,        /* no device / CUDA runtime error (see miqp_b200_last_error) */
  MIQP_B200_ERR_ARG = -2,         /* malformed problem or argument */
  MIQP_B200_ERR_UNSUPPORTED = -3, /* shape outside what the kernels are built for */
  MIQP_B200_ERR_RESOURCE = -4     /* (unused since pool exhaustion is reported per plan: MiqpB200SolveInfo.pool_exhausted) */
};

/* OptimizationStatus of the reference (src/cplex_wrapper.hpp:54-59) */
enum {
  MIQP_B200_SUCCESS = 0,
  MIQP_B200_FAILED_NO_SOLUT = 1,
  MIQP_B200_FAILED_SEG_FAULT = 2,
  MIQP_B200_FAILED_TIMEOUT = 3
};

/* One MIQP instance: the content of ModelParameters, row-major, host memory.
 * Index conventions: cars c in [0,C), steps i in [0,N), regions j in [0,R). */
typedef struct MiqpB200Problem {
  int N, R, C, O, L, E;       /* NumSteps, nr_regions, NumCars, nr_obstacles, max_lines_obstacles, nr_environments */
  double ts;
  double min_vel, max_vel, total_min_acc, total_max_acc, total_min_jerk, total_max_jerk;
  double maximum_slack, w_slack, w_slack_obs, min_region_change_speed;
  double gap_tol, time_limit; /* relative_mip_gap_tolerance, max_solution_time */
  const double *safety;        /* [N]  agent_safety_distance */
  const double *safety_slack;  /* [N]  agent_safety_distance_slack */
  const double *w_pos_x, *w_vel_x, *w_acc_x, *w_pos_y, *w_vel_y, *w_acc_y, *w_jerk_x, *w_jerk_y; /* [C] */
  const double *wheelbase, *radius;                 /* [C] */
  const double *x0;                                 /* [C][6] x,vx,ax,y,vy,ay (IntitialState) */
  const double *x_ref, *vx_ref, *y_ref, *vy_ref;    /* [C][N] */
  const double *min_acc_x, *max_acc_x, *min_acc_y, *max_acc_y;     /* [C][R] */
  const double *min_jerk_x, *max_jerk_x, *min_jerk_y, *max_jerk_y; /* [C][R] */
  const int *initial_region;   /* [C], 1-based as in ModelParameters */
  const int *possible_region;  /* [C][R] */
  const double *obs_edges;     /* [O][N][L][4] x1,y1,x2,y2 of ObstacleConvexPolygon[o][i] */
  const int *obs_nedges;       /* [O][N] */
  const int *obs_soft;         /* [O] */
  const double *env_edges;     /* [env_off[E]][4] edges of MultiEnvironmentConvexPolygon */
  const int *env_off;          /* [E+1] */
  const double *frac;          /* [R][4] fraction_parameters */
  const double *poly_sint_ub, *poly_sint_lb, *poly_coss_ub, *poly_coss_lb; /* [R][3] */
  const double *poly_kappa_max, *poly_kappa_min;                           /* [R][3] */
} MiqpB200Problem;

/* Column layout = decision_variables.mod order.  Blocks 0..11 are u_x,u_y,pos_x,vel_x,
 * acc_x,pos_y,vel_y,acc_y,pos_x_front_UB,pos_x_front_LB,pos_y_front_UB,pos_y_front_LB,
 * each [C][N]; then notWithinEnvironment{Rear,FrontUbUb,FrontLbUb,FrontUbLb,FrontLbLb}
 * [5][C][E][N]; active_region [C][N][R]; region_change_not_allowed_{x_positive,y_positive,
 * x_negative,y_negative,combined} [5][C][N]; deltacc [C][O][N][L]; deltacc_front
 * [C][O][N][L][4]; slackvarsObstacle [C][O][N]; slackvarsObstacle_front [C][O][N][4];
 * car2car_collision [K][K][N][16]; slackvars [K][K][N][4], K = C-1. */
typedef struct MiqpB200Layout {
  int C, N, R, O, L, E, K;
  int base_nwe, base_ar, base_rcna, base_dcc, base_dcf, base_so, base_sof, base_c2c, base_sv;
  int ncols;
} MiqpB200Layout;

/* SolutionProperties statistics (src/cplex_wrapper.hpp:41-52, filled at :680-690) */
typedef struct MiqpB200Sizes {
  int ncols, ncont, nbin;
  long nrows, nnz_struct, nnz; /* nnz excludes exact-zero coefficients, as CPLEX counts */
} MiqpB200Sizes;

typedef struct MiqpB200SolveInfo {
  int status;            /* MIQP_B200_SUCCESS / FAILED_NO_SOLUT / FAILED_TIMEOUT */
  int proven;            /* 1 if gap <= gap_tol was reached */
  double objective, best_bound, gap; /* gap = |best_bound-objective| / (1e-10+|objective|) */
  double seconds;        /* solve time of THIS plan: host clock (from the start of the batch) at the end of the round after which the plan was
                          * finished or hit its own time_limit; the batch's wall time for a plan that was stopped with the batch */
  double max_violation;  /* of the returned vector against the full big-M model, device-evaluated */
  long nodes, qp_iters, rounds;
  long uncertified;      /* node relaxations closed without optimum, feasible point or Farkas certificate; their bounds stay in best_bound */
  int pool_exhausted;    /* 1: the node pool of this plan ran out (children were dropped, their bound stays in best_bound; result not proven) */
} MiqpB200SolveInfo;

typedef struct MiqpB200Options {
  int device;            /* CUDA ordinal */
  int nodes_per_round;   /* max node relaxations taken from one plan's frontier per round; 0 = auto */
  int pool_capacity;     /* open-node slots per plan; 0 = auto */
  int max_rounds;        /* 0 = unlimited (time limit still applies) */
  int verbose;
} MiqpB200Options;

typedef struct MiqpB200Solver MiqpB200Solver;

const char *miqp_b200_version(void);
void miqp_b200_default_options(MiqpB200Options *opt);
int miqp_b200_create(const MiqpB200Options *opt, MiqpB200Solver **out);
void miqp_b200_destroy(MiqpB200Solver *s);
const char *miqp_b200_last_error(const MiqpB200Solver *s);

/* host-only, closed form */
int miqp_b200_layout(const MiqpB200Problem *p, MiqpB200Layout *out);

/* Device row instantiation.  Counts first (any output pointer may be NULL); the CSR is in
 * OPL instantiation order with structural zeros kept: rowptr[nrows+1], cols/vals[nnz_struct],
 * lo/hi[nrows] (+-HUGE_VAL for one-sided rows). */
int miqp_b200_sizes(MiqpB200Solver *s, const MiqpB200Problem *p, MiqpB200Sizes *out);
int miqp_b200_assemble(MiqpB200Solver *s, const MiqpB200Problem *p, long *rowptr, int *cols,
                       double *vals, double *lo, double *hi);

/* Row instantiation of a whole batch into device-resident CSR buffers (kept by the solver), `repeats` timed passes after one
 * untimed pass: average kernel time in ms (CUDA events), total rows and structural non-zeros.  What opl.generate()
 * (reference src/cplex_wrapper.cpp:98) does per plan, measured for the roofline of the assembly kernel. */
int miqp_b200_assemble_batch(MiqpB200Solver *s, const MiqpB200Problem *problems, int count, int repeats,
                             float *device_ms, long *rows, long *nnz_struct);

/* objective and max violation (rows, bounds, integrality) of a full column vector */
int miqp_b200_evaluate(MiqpB200Solver *s, const MiqpB200Problem *p, const double *x,
                       double *objective, double *max_violation);

/* Solve `count` independent plans.  warm[k] (may be NULL, as may `warm`) is a full column
 * vector used as MIP start; x_out[k] receives ncols(k) doubles; infos[k] the status. */
int miqp_b200_solve_batch(MiqpB200Solver *s, const MiqpB200Problem *problems, int count,
                          const double *const *warm, double *const *x_out,
                          MiqpB200SolveInfo *infos);

/* The same in three steps, for callers that keep the batch resident in HBM:
 * upload (H2D, tables, initial frontier) / run (device only; may be repeated, every run
 * restarts from the uploaded state) / fetch (D2H). */
int miqp_b200_batch_upload(MiqpB200Solver *s, const MiqpB200Problem *problems, int count,
                           const double *const *warm);
/* Receding-horizon replanning (reference: MiqpPlanner::CalculateWarmstart + EnvironmentWarmstart, src/miqp_planner.cpp:787-1115, and the MIP
 * start of src/cplex_wrapper.cpp:494-639): upload of the NEXT planning cycle of the plans of the previous batch on this solver
 * (same count, order and shapes; states, references and obstacle predictions advanced by the caller).  The MIP start of every plan
 * is its previous incumbent shifted by one step ON THE DEVICE -- no solution vector crosses PCIe; plans without a previous
 * incumbent, or whose shape changed, start cold. */
int miqp_b200_batch_upload_replan(MiqpB200Solver *s, const MiqpB200Problem *problems, int count);
int miqp_b200_batch_run(MiqpB200Solver *s, float *device_ms);
int miqp_b200_batch_fetch(MiqpB200Solver *s, double *const *x_out, MiqpB200SolveInfo *infos);

/* Streaming run: the same search as batch_run (after batch_upload or batch_upload_replan; batch_fetch, batch_fetch_compact,
 * fetch_vector, pool_sizes and pool_fetch return the same afterwards), but every plan is handed to `on_done` as soon as its
 * search ends instead of when the batch ends.  The device harvests a plan in the round in which it is marked finished (its
 * result is final then); the callback runs on the calling thread, between rounds, at most one round later, in ascending k
 * within a round.  Plans still searching when the batch stops (time limit, max_rounds), and plans whose own time limit was over
 * before the first round, are delivered at the end.  Every plan is delivered exactly once.
 * `traj` ([C][N][8], the compact layout of batch_fetch_compact) and `info` are valid during the call only.  `info` equals what
 * batch_fetch_compact returns for plan k after the run, except `rounds`: the rounds the batch had run when the plan finished
 * (the batch's rounds for the plans delivered at the end).  The callback must not call into this solver.
 * ERR_ARG: on_done == NULL or no upload. */
typedef void (*MiqpB200PlanDone)(void *user, int k, const double *traj, const MiqpB200SolveInfo *info);
int miqp_b200_batch_run_streaming(MiqpB200Solver *s, MiqpB200PlanDone on_done, void *user, float *device_ms);

/* Compact results: per plan the trajectory of every car, [C][N][8] doubles (pos_x, vel_x, acc_x, pos_y, vel_y, acc_y, u_x, u_y per
 * step: what MiqpPlanner::GetTrajectory reads, src/miqp_planner.cpp:1117-1192) instead of the full OPL column vector (config 2:
 * 2.5 kB instead of 33 kB per plan across PCIe).  Objective, gap, status and violation in `infos` are those of the full vector,
 * which stays on the device until the next upload: fetch_vector(s, k, x_out) copies plan k's RawResults vector on demand, and
 * batch_upload_replan uses the incumbents in place. */
int miqp_b200_batch_fetch_compact(MiqpB200Solver *s, double *const *traj_out, MiqpB200SolveInfo *infos);
int miqp_b200_fetch_vector(MiqpB200Solver *s, int k, double *x_out /* [ncols of plan k] */);
int miqp_b200_solve_batch_compact(MiqpB200Solver *s, const MiqpB200Problem *problems, int count, const double *const *warm,
                                  double *const *traj_out, MiqpB200SolveInfo *infos);

/* The same search in steps, for a caller that shards the FRONTIER of the uploaded plans over several GPUs (one process and one
 * solver per GPU; SURVEY section 8(e).2).  Every rank uploads the same batch and runs the same deterministic ramp-up
 * (frontier_start, frontier_rounds); frontier_split then keeps, in every open list, the nodes whose uid hashes to this rank.
 * From there on only incumbent OBJECTIVES travel: frontier_get_ub -> min-allreduce (8 bytes per plan) -> frontier_tighten
 * (host buffers), or an in-place NCCL min-allreduce on frontier_ub_device, every few rounds.  frontier_finish + batch_fetch return this rank's own incumbent (status FAILED_NO_SOLUT if it has none) and
 * the best bound of its share; the caller takes the minimum of both over the ranks and broadcasts the winner's vector. */
int miqp_b200_frontier_start(MiqpB200Solver *s);
int miqp_b200_frontier_rounds(MiqpB200Solver *s, int nrounds, int *unfinished_plans);
int miqp_b200_frontier_split(MiqpB200Solver *s, int rank, int world);
/* fingerprint of every open list (call on every rank after the ramp-up and compare: the split is only sound if the ramp-ups agree) */
int miqp_b200_frontier_fingerprint(MiqpB200Solver *s, long long *fp /* [count] */);
/* device address of the incumbent objectives ([count] doubles on the solver's GPU): an in-place ncclAllReduce(min) on it is the
 * whole exchange (no host copy); synchronise the communication stream before the next frontier_rounds */
int miqp_b200_frontier_ub_device(MiqpB200Solver *s, void **ub, int *count);
int miqp_b200_frontier_get_ub(MiqpB200Solver *s, double *ub /* [count] */);
int miqp_b200_frontier_tighten(MiqpB200Solver *s, const double *ub /* [count] */);
int miqp_b200_frontier_finish(MiqpB200Solver *s, float *device_ms);

/* Solution pool (CPLEX's pool, counted by SolutionProperties.NrSolutionPool): up to `capacity` distinct integer-feasible
 * completions per plan that the search solved, best first.  0 = off (default); 1..64; takes effect at the next upload.
 * The pool records leaves the search solves anyway (those that do not beat the incumbent too); it does not change the search or
 * its results.  Policy: the `capacity` best leaves by the incumbent's key (search value, node uid) with pairwise different
 * decisions, so the pool is as deterministic as the search.  The pool of the last run stays on the device until the next upload. */
int miqp_b200_set_solution_pool(MiqpB200Solver *s, int capacity);
typedef struct MiqpB200PoolEntry {
  double objective, max_violation; /* of the expanded full vector, device-evaluated, like MiqpB200SolveInfo */
  double search_value;             /* value the search stored (order key with uid) */
  int converged;                   /* 1: the leaf QP was solved to optimality */
  int round;                       /* round of the search that solved the leaf */
  unsigned long long uid;          /* node uid */
} MiqpB200PoolEntry;
/* entries per plan, [count]; ERR_ARG with the pool off or before a run */
int miqp_b200_pool_sizes(MiqpB200Solver *s, int *sizes /* [count] */);
/* the first min(size, max_entries) entries of plan k in (search_value, uid) order -- entry 0 is the incumbent; after pool_merge it
 * is the best merged entry, which is the combined incumbent of the ranks, not necessarily this rank's own --, their full column
 * vectors (x_out, RawResults order like fetch_vector) and trajectories (traj_out, the compact layout of batch_fetch_compact) */
int miqp_b200_pool_fetch(MiqpB200Solver *s, int k, int max_entries, MiqpB200PoolEntry *entries,
                         double *x_out /* [max_entries][ncols(k)] or NULL */,
                         double *traj_out /* [max_entries][C][N][8] or NULL */, int *n_out);
/* Pools of a frontier-sharded search (frontier_*): each rank's pool holds the leaves that rank solved.  After frontier_finish every
 * rank exports its pool, the exports are all-gathered (NCCL in place on the device buffers, or through the host), and every rank
 * merges them: the result is the pool of the union of all ranks' leaves, the same on every rank and for any rank order.
 * export: packs this solver's pool into a solver-owned device buffer (*dev, *bytes; valid until the next export, upload or
 * destroy).  Layout: a 64-byte header (magic/version, count, capacity, zstride, ndec_stride, hash of every plan's C, N, R, O, L,
 * E, ncols), then cnt[count], rec[count][cap], dec[count][cap][ndec_stride], z[count][cap][zstride], sections 16-byte aligned.
 * merge: `gathered` holds `world` exports back to back (world x bytes; host memory or device memory); it replaces this solver's
 * pool by the capacity best entries by (search_value, uid) with pairwise different decisions over all of them.  pool_sizes and
 * pool_fetch then return the merged pool; entries are expanded and evaluated on this rank's own copy of the problem data.
 * ERR_ARG, the pool unchanged: no run, pool off, world < 1, world x capacity > 512, or a header that does not match this
 * solver's upload (another capacity or batch shape). */
int miqp_b200_pool_export(MiqpB200Solver *s, void **dev, size_t *bytes);
int miqp_b200_pool_merge(MiqpB200Solver *s, const void *gathered, int world);

/* counters of the last run: kernel launches, node relaxations, IPM iterations, seconds
 * spent in the node kernel (CUDA events on the solver stream) */
typedef struct MiqpB200RunStats {
  long launches, node_kernel_launches, nodes, qp_iters, rounds;
  double node_kernel_ms, total_ms;
  long h2d_bytes, d2h_bytes;
  long rows_visited;     /* sum over node relaxations and IPM iterations of active rows */
  double pack_ms, upload_ms, fetch_ms; /* host wall time of the last batch: flatten into the staging blobs / H2D + tables + pool setup / D2H + scatter */
} MiqpB200RunStats;
int miqp_b200_run_stats(const MiqpB200Solver *s, MiqpB200RunStats *out);

/* Device time over several runs, also of several solvers of one GPU that work concurrently (two batches in flight on two
 * streams): mark(s, 0) / mark(s, 1) record CUDA events on the solver's stream; elapsed(from, to) = time from mark 0 of `from` to
 * mark 1 of `to` (both events are waited for). */
int miqp_b200_mark(MiqpB200Solver *s, int which);
int miqp_b200_elapsed(MiqpB200Solver *from, MiqpB200Solver *to, float *ms);

/* Diagnostics of the last run (zeros unless the library was built with -DMQ_PROF):
 * out256[0..100] histogram of interior-point iterations per node relaxation, out256[128..131]
 * clock64 cycles in row passes / Riccati factorisation / vector sweeps / whole node solves,
 * out256[132..133] infeasible node relaxations and their iterations. */
int miqp_b200_debug_profile(MiqpB200Solver *s, unsigned long long *out256);
/* -DMQ_PROF builds: per-iteration (alpha, mu, primal residual, sigma, lambda max) of up to 8 slow node relaxations, [8][512] */
int miqp_b200_debug_traces(MiqpB200Solver *s, double *out4096);

/* FP64 FMA throughput of the device in TFLOP/s (DFMA micro-benchmark, best of 5): the
 * roofline denominator of the node kernel, which MEASURED_PEAKS.json does not provide. */
int miqp_b200_measure_fp64_peak(MiqpB200Solver *s, double *tflops);

#ifdef __cplusplus
}
#endif
#endif
