// kernels.cuh -- launcher declarations shared by the host driver (solver.cu).
#pragma once
#include "dev_problem.cuh"

namespace miqp {

// ---- formulation.cu -------------------------------------------------------------------
void launch_prepare_tables(DevProb *probs, double *dblob, int *iblob, int count, cudaStream_t st);
void launch_assemble_rows(const DevProb *probs, const double *dblob, const int *iblob, int count, long max_rows,
                          long *rowptr, int *cols, double *vals, double *lo, double *hi,
                          unsigned long long *nnz_count, cudaStream_t st);
void launch_evaluate(const DevProb *probs, const double *dblob, const int *iblob, int count, long max_rows,
                     const double *xall, double *max_viol, double *objective, cudaStream_t st);
// the same for the plans list[0 .. *n) only; *n is read on the device, max_n (>= *n) sizes the grid.  max_viol[list[e]] must be
// zeroed before (bnb_harvest_kernel does it)
void launch_evaluate_list(const DevProb *probs, const double *dblob, const int *iblob, const int *list, const int *n, int max_n,
                          long max_rows, const double *xall, double *max_viol, double *objective, cudaStream_t st);

// ---- bnb.cu ---------------------------------------------------------------------------
// entry of the solution pool (BnbState::pool_rec)
struct PoolRec {
  double val;               // value the search stored for the leaf (the incumbent's ub when it is the best)
  unsigned long long uid;   // node uid (tie break, as inc_uid)
  int round, converged;     // round the leaf was solved in; 1 if its QP was solved to optimality
};

// Device-resident branch and bound state of a batch of plans.
struct BnbState {
  int count;            // plans
  int cap;              // node slots per plan
  int ndec_stride;      // bytes per node decision vector (max over plans, multiple of 16)
  int zstride;          // doubles per incumbent trajectory (max C*N*8 + 4*P*N)
  int kmax;             // row slots per stage (max over plans)
  int npad;             // stages padded to a multiple of 32 (max over plans)
  int nwarps;           // node relaxations in flight (resident teams of the node kernel)
  int sel_per_plan;     // stride of sel_idx: most node relaxations a plan may take in one round
  int sel_base;         // nodes per plan per round once an incumbent exists (raised when few plans are active)
  int sel_dive;         // nodes per plan per round while diving for the first incumbent
  int dive_fill;        // >0: while diving, widen to (resident warps / active plans) / dive_fill heads when few plans are active
  int multi_heur;                   // multi-car plans without incumbent: completion heuristic at every multi_heur-th level of the tree (0: off)
  int dive_patience, dive_growth;   // a plan without incumbent after dive_patience rounds widens its dive by dive_growth heads per round
  int work_cap;
  int force_multi;      // route every plan to the CTA-per-node kernel (test hook)
  // node pools [count][cap]
  unsigned char *dec;
  double *bound;
  int2 *meta;           // depth, rank
  unsigned long long *uid;
  int *open_idx; int *open_cnt;
  int *free_stack; int *free_cnt;
  int *sel_idx; int *sel_cnt;      // slots handed to the node kernel in the last round [count][sel_per_plan]
  unsigned long long *keybuf;      // [count][cap]
  // suspended relaxations: a node whose interior-point solve exceeds its iteration budget is parked with its state and
  // continues in the next round (two pools, written alternately; susp_slot = index in the pool of the round that parked it)
  double *susp_pool[2]; int *susp_slot; int *susp_cnt; int susp_slots; long susp_stride; int susp_budget;
  double *zpool;        // [count][cap][zp_stride] relaxed optimum of the parent (warm start of the child's interior-point solve); null = off
  int zp_stride;
  double warm_mu;       // complementarity target of the warm start
  double tau_k;         // step fraction to the boundary = max(0.995, 1 - tau_k * mu); 0 = constant 0.995
  // per plan
  double *ub;           // incumbent objective (inf if none)
  double *cutoff;       // snapshot used by the node kernel in the current round
  double *pruned_lb;
  int *done;               // 0 searching, 1 finished (frontier exhausted within the gap), 2 stopped at its own time limit,
                           // 3 stopped on the caller's request (stop)
  int *done_round;         // round in which the plan finished (its solve time = the host's clock at that round)
  const double *tlimit;    // per-plan time limits in seconds (device copy)
  int *lock;
  double *inc_z;        // [count][zstride]
  unsigned char *inc_dec;  // [count][ndec_stride]
  unsigned long long *inc_uid;  // tie break between equal incumbents (deterministic result)
  unsigned long long *stat_nodes, *stat_iters, *stat_rows;
  unsigned long long *stat_uncert;   // node relaxations closed without optimum, feasible point or infeasibility certificate
  int *overflow;                     // per plan: 1 if its node pool ran out (children dropped, bound kept in pruned_lb)
  double *dbg;                // [-DMQ_PROF] per-CTA iteration traces [ctas + 8][512]; slots ctas.. hold the claimed slow relaxations
  unsigned long long *prof;   // [256] diagnostics (filled only by -DMQ_PROF builds): [it] histogram of IPM iterations per node, [128..] cycles
  // round control
  int2 *work; int *work_cnt; int *work_next; int *active; int *err; int *active_prev;
  int2 *work2; int *work_cnt2; int *work_next2;   // plans with NumCars > 1 (bnb_multi.cu)
  // solution pool (pool_cap > 0): the pool_cap best distinct leaves of every plan by the incumbent's key (value, uid), unsorted;
  // records laid out like the incumbent's (inc_z, inc_dec).  Written under the plan's lock by pool_insert (bnb_common.cuh).
  int pool_cap;
  double *pool_z;           // [count][pool_cap][zstride]
  unsigned char *pool_dec;  // [count][pool_cap][ndec_stride]
  PoolRec *pool_rec;        // [count][pool_cap]
  int *pool_cnt;            // [count]
  // streaming runs (miqp_b200_batch_run_streaming): 1 once a finished plan's result has been harvested; null otherwise
  int *delivered;           // [count]
  // stop requests of the caller (miqp_b200_request_stop): nonzero = select stops the plan; null while the run has none
  const unsigned char *stop;   // [count]
};

// one plan's share of the solution pool, handed to the out-of-line insertion (kernel parameters stay in parameter space)
struct PoolRef {
  double *z; unsigned char *dec; PoolRec *rec; int *cnt;
  int cap, zstride, ndec_stride;
};

void launch_bnb_init(const BnbState &st, const DevProb *probs, const unsigned char *warm_dec /* [count][ndec_stride] or null */,
                     const int *has_warm, cudaStream_t s);
void launch_bnb_select(const BnbState &st, const DevProb *probs, int round, double elapsed_s, cudaStream_t s);
constexpr int SUSP_REQUEUE = 1 << 30;      // susp_slot mark of a node that is solved again from the cold start (keeps its slot like a parked one)
constexpr int NODE_TEAM_WARPS = 4;        // warps that share one node relaxation (bnb_nodes_kernel), 2 teams per SM
constexpr int NODE_TEAMS_PER_SM = 2;      // 255 registers per thread; 3 (168 registers, spills) gave no gain: profiles/r1k, r2_knobs_heldout
constexpr int NODE_TEAM_WARPS_NARROW = 2; // throughput variant: two warps per node, four teams per SM (rounds with more nodes than the four-warp teams hold)
constexpr int NODE_TEAM_WARPS_WIDE = 8;   // the same for rounds with fewer nodes than SMs, 1 team per SM
// returns 0 or a cudaError
int launch_bnb_nodes(const BnbState &st, const DevProb *probs, const double *dblob, const int *iblob,
                     int smem_per_warp, int warps_per_cta, int ctas, int maxN, int row_np, int round, cudaStream_t s);
void launch_bnb_split(const BnbState &st, int rank, int world, cudaStream_t s);       // frontier sharding: keep this rank's share of every open list
void launch_bnb_shift_warm(const DevProb *probs, const int *iblob, int count, const unsigned char *prev_dec, int prev_stride, const double *prev_ub,
                           const unsigned long long *prev_uid, const int *same_shape, unsigned char *warm_dec, int stride, int *has_warm, cudaStream_t s);
void launch_bnb_fingerprint(const BnbState &st, unsigned long long *out, cudaStream_t s);   // frontier sharding: open-list fingerprint per plan
void launch_bnb_tighten(const BnbState &st, const double *ub, cudaStream_t s);      // st.ub = min(st.ub, ub): incumbents of other ranks
void launch_bnb_finish(const BnbState &st, const DevProb *probs, const double *dblob, const int *iblob,
                       double *xall, double *best_bound, cudaStream_t s);
// full column vectors of n pool entries of plan k: block e expands entry idx[e] with eprobs[e] (plan k's DevProb, x_base = e * ncols)
// into xall; the entry's trajectory goes to zs[e * zstride] (pool storage is not modified)
void launch_pool_expand(const BnbState &st, int k, const int *idx, int n, const DevProb *eprobs, const double *dblob, const int *iblob,
                        double *zs, double *xall, cudaStream_t s);
// byte offsets of the sections of one pool export (miqp_b200_pool_export): header, cnt[count], rec[count][pool_cap],
// dec[count][pool_cap][ndec_stride], z[count][pool_cap][zstride]; every section and the whole export 16-byte aligned
struct PoolExportLayout { long off_cnt, off_rec, off_dec, off_z, bytes; };
constexpr int POOL_MERGE_MAX = 512;   // candidates per plan (world x pool_cap) pool_merge_kernel sorts in shared memory
// this solver's pool := the pool_cap best entries, by (value, uid), with pairwise different decisions (the plan's ndec_pad bytes)
// of `world` exports stored back to back at `gathered` (device memory of the solver's GPU, exports lay.bytes apart; the pool
// storage itself is not read)
void launch_pool_merge(const BnbState &st, const DevProb *probs, const unsigned char *gathered, const PoolExportLayout &lay, int world,
                       cudaStream_t s);
// ---- streaming runs: per-round harvest of the plans that select marked finished -------------------------------------------
// one record per harvested plan, then its trajectory [C][N][8] (inc_z after expand_solution); records are rec_stride doubles apart
struct StreamRec {
  double objective, max_violation, best_bound, ub;                     // evaluate_kernel's values, bnb_finish's best bound, incumbent
  unsigned long long inc_uid, nodes, iters, rows, uncert;              // incumbent uid and the four stats counters
  int k, done, done_round, overflow;                                   // plan index and its search state
};
constexpr int STREAM_REC_HDR = 12;   // doubles before the trajectory
constexpr int HARVEST_GRID = 1024;   // most blocks of a harvest kernel (they stride over the harvested plans)
static_assert(sizeof(StreamRec) <= STREAM_REC_HDR * sizeof(double), "StreamRec outgrew its header");
// plans to harvest in ascending order into list[0 .. *n): finished (done != 0) and not yet delivered -- or, with all = 1, every
// plan not yet delivered (end of the run); marks them delivered and zeroes their max_viol for launch_evaluate_list
void launch_bnb_harvest(const BnbState &st, int all, int *list, int *n, double *max_viol, cudaStream_t s);
// finishing of the harvested plans (best bound, full column vector into xall, exact trajectory in inc_z)
void launch_bnb_harvest_finish(const BnbState &st, const DevProb *probs, const double *dblob, const int *iblob, const int *list,
                               const int *n, int max_n, double *xall, double *best_bound, cudaStream_t s);
// records of the harvested plans into out[e * rec_stride]
void launch_bnb_harvest_pack(const BnbState &st, const DevProb *probs, const int *list, const int *n, int max_n, const double *obj,
                             const double *viol, const double *best_bound, double *out, long rec_stride, cudaStream_t s);
// ---- anytime runs: per-round harvest of the plans whose incumbent changed -----------------------------------------------------
// one record per plan, then its trajectory [C][N][8] (a scratch copy of inc_z after expand_solution); records rec_stride doubles apart
struct IncRec {
  double objective, max_violation, ub, best_bound;   // evaluate_kernel's values of the expanded incumbent, its search value, best bound
  unsigned long long inc_uid, nodes, iters;          // incumbent uid, node and interior-point iteration counters so far
  int k, round;                                      // plan index, round the incumbent was found in
};
constexpr int INC_REC_HDR = 8;   // doubles before the trajectory
static_assert(sizeof(IncRec) <= INC_REC_HDR * sizeof(double), "IncRec outgrew its header");
// plans whose incumbent changed since the last delivery (inc_uid != reported_uid), ascending, into list[0 .. *n); sets
// reported_uid and zeroes their max_viol for launch_evaluate_list
void launch_bnb_inc_list(const BnbState &st, unsigned long long *reported_uid, int *list, int *n, double *max_viol, cudaStream_t s);
// the listed incumbents expanded in a scratch copy of inc_z (zs[s * zstride]; inc_z is not modified) into xall, and every listed
// plan's best bound (open nodes, the nodes select handed to this round's node kernels if with_sel, pruned_lb, at most ub) into
// best_bound
void launch_bnb_inc_expand(const BnbState &st, const DevProb *probs, const double *dblob, const int *iblob, const int *list,
                           const int *n, int max_n, int with_sel, double *zs, double *xall, double *best_bound, cudaStream_t s);
// records of the listed plans into out[e * rec_stride]; `round`: the round whose select has just run
void launch_bnb_inc_pack(const BnbState &st, const DevProb *probs, const int *list, const int *n, int max_n, const double *obj,
                         const double *viol, const double *best_bound, const double *zs, int round, double *out, long rec_stride,
                         cudaStream_t s);
// ---- frontier sharding with incumbent deliveries (miqp_b200_frontier_inc_export / _merge) -----------------------------------
// One rank's export block: a 64-byte header, then per plan its best bound (double), node and interior-point iteration counters
// (unsigned long long) and stop request (byte), each section 16-byte aligned (together: the summary), then n_records records of
// rec_stride doubles, IncRec + trajectory [C][N][8] as launch_bnb_inc_pack writes them, in ascending plan order.
struct FrontierIncHeader {
  unsigned magic, version;
  int count, n_records;
  long rec_stride;                 // doubles per record
  long rounds;                     // rounds this rank had run at the export
  unsigned long long shape_hash;   // FNV-1a over (C, N, R, O, L, E, ncols) of every plan, as the pool export
  unsigned char pad[24];
};
static_assert(sizeof(FrontierIncHeader) == 64, "frontier export header size");
struct FrontierIncLayout { long off_bb, off_nodes, off_iters, off_stop, summary_bytes, rec_stride; };
// one merged delivery: the winning record with the merged best bound and the counters summed over the ranks, and the winner's
// rank; then its trajectory.  Records FI_OUT_HDR + C * N * 8 doubles apart (out_stride)
struct FrontierIncOut {
  IncRec r;
  int rank, pad_;
};
constexpr int FI_OUT_HDR = 10;   // doubles before the trajectory
static_assert(sizeof(FrontierIncOut) <= FI_OUT_HDR * sizeof(double), "FrontierIncOut outgrew its header");
// summary of this rank into block (best bounds with no unsolved selected nodes, counters); the header and stop bytes come from
// the host
void launch_frontier_inc_summary(const BnbState &st, unsigned char *block, const FrontierIncLayout &lay, cudaStream_t s);
// merge of `world` blocks block_bytes apart at g (device memory): per plan the best record by (objective, rank); delivered, in
// ascending plan order into list / out (headers) / src (rank, record), if its key is below (key_obj, key_rank) (key_rank < 0:
// nothing delivered yet), which it then becomes.  stop_out = OR of the ranks' stop bytes.  *n = deliveries.
void launch_frontier_inc_merge(const BnbState &st, const unsigned char *g, const FrontierIncLayout &lay, long block_bytes, int world,
                               double *key_obj, int *key_rank, unsigned char *stop_out, int *list, int2 *src, int *n, double *out,
                               long out_stride, cudaStream_t s);
// trajectories of the deliveries into out[e * out_stride + FI_OUT_HDR]
void launch_frontier_inc_pack(const DevProb *probs, const unsigned char *g, const FrontierIncLayout &lay,
                              long block_bytes, const int *list, const int2 *src, const int *n, int max_n, double *out, long out_stride,
                              cudaStream_t s);
int node_kernel_smem_per_warp(int maxN, int kmax, int ndec_stride);
int node_kernel_narrow_np(int N);                                  // row stride of the (s, lambda) records of a two-warp team
int node_kernel_smem_narrow(int N, int kmax, int ndec_stride);   // shared memory of a two-warp team (uniform horizon N)
int node_kernel_max_ctas(int smem_per_cta, int threads);

// ---- bnb_multi.cu ---------------------------------------------------------------------
// CTA-per-node kernel for plans with several cars.  ws_bytes = workspace of one node (max over the
// plans of the batch); it lives in shared memory when it fits, else in gws[ctas][ws_bytes].
long multi_workspace_bytes(int C, int N, int P, int kmax, int ndec_stride);
int multi_kernel_max_ctas(int smem_bytes, int threads);
int launch_bnb_nodes_multi(const BnbState &st, const DevProb *probs, const double *dblob, const int *iblob,
                           double *gws, long ws_bytes, int use_smem, int threads, int ctas, int round, cudaStream_t s);

}  // namespace miqp
