// solver.cu -- host driver and C ABI (include/miqp_b200.h) of the B200 MIQP backend.
//
// Host responsibilities (everything else runs on the device):
//   * flatten a batch of plans (ModelParameters, reference src/miqp_planner_data.hpp:99-185)
//     into one double blob + one int blob and upload them with one copy each;
//   * the two scalar pre-computations OPL does in its `execute` blocks
//     (cplexmodel/initialization.mod:16-29: front axle point at step 1 from atan2/cos/sin)
//     and the list of mode alternatives per car;
//   * MIP start: decisions of a full column vector (src/cplex_wrapper.cpp:494-639);
//   * the round loop: launch select + node kernels, poll the number of unfinished plans,
//     enforce the time limit (tilim, cplexmodel.mod:8-10).
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <thread>
#include <algorithm>
#include <vector>

#include "../../include/miqp_b200.h"
#include "kernels.cuh"
#define MIQP_PINNED_BLOBS 1
#include "host_pack.hpp"

using namespace miqp;
using namespace miqp::hostpack;
namespace miqp { double measure_fp64_tflops(int num_sms, cudaStream_t st, int reps); }

namespace {

#define CK(call)                                                                         \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      char buf_[512];                                                                    \
      snprintf(buf_, sizeof buf_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      throw std::runtime_error(buf_);                                                    \
    }                                                                                    \
  } while (0)

template <class T>
struct DevBuf {
  T *p = nullptr;
  size_t n = 0;
  void ensure(size_t count) {
    if (count <= n) return;
    if (p) cudaFree(p);
    p = nullptr; n = 0;
    CK(cudaMalloc(&p, count * sizeof(T)));
    n = count;
  }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  ~DevBuf() { release(); }   // (every buffer of a solver goes with it, also those miqp_b200_destroy does not list)
};

}  // namespace

struct MiqpB200Solver {
  MiqpB200Options opt;
  std::string err;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evr0 = nullptr, evr1 = nullptr;
  cudaEvent_t mark[2] = {nullptr, nullptr};   // miqp_b200_mark / miqp_b200_elapsed: device time across several runs and solvers
  int num_sms = 0;
  // batch
  Packed pk;
  std::vector<hostpack::PackedLocal> pack_parts;
  std::vector<double> time_limits;
  DevBuf<DevProb> d_probs;
  DevBuf<double> d_dblob;
  DevBuf<int> d_iblob;
  DevBuf<double> d_x, d_viol, d_obj, d_bb;
  DevBuf<long> a_rowptr; DevBuf<int> a_cols; DevBuf<double> a_vals, a_lo, a_hi; DevBuf<unsigned long long> a_cnt;   // assembled big-M model (kept between calls)
  DevBuf<unsigned char> d_warm;
  DevBuf<int> d_haswarm;
  std::vector<unsigned char> h_warm;
  std::vector<int> h_haswarm;
  bool any_warm = false;
  // bnb state buffers
  BnbState st;
  DevBuf<unsigned char> b_dec, b_incdec;
  DevBuf<double> b_bound, b_ub, b_cutoff, b_pruned, b_incz, b_zpool, b_dbg, b_susp0, b_susp1;
  DevBuf<int> b_suspslot, b_suspcnt;
  DevBuf<int2> b_meta, b_work;
  DevBuf<unsigned long long> b_uid, b_keybuf, b_incuid, b_stats, b_prof;
  DevBuf<int> b_open, b_opencnt, b_free, b_freecnt, b_sel, b_selcnt, b_done, b_lock, b_ctrl, b_overflow;
  int smem_per_warp = 0, warps_per_cta = 4, ctas = 0, wide_ctas = 0;
  int narrow_ctas = 0, smem_narrow = 0, narrow_np = 0, narrow_min = 0; long narrow_launches = 0;   // two-warp teams (throughput rounds)
  // CTA-per-node kernel for plans with several cars
  int n_single = 0, n_multi = 0, multi_threads = 64, multi_ctas = 0, multi_use_smem = 1;
  long multi_ws_bytes = 0;
  DevBuf<double> b_multi_ws;
  DevBuf<int2> b_work2;
  bool uploaded = false, ran = false;
  // the current run (start_run .. finish_run, batch runs and the stepped frontier search alike)
  long fr_rounds = 0; int fr_ctrl0 = 0;                       // rounds run so far / work items of the last round
  std::chrono::steady_clock::time_point fr_t0;                // start of the run (time limit)
  long fr_launches = 0, fr_node_launches = 0; double fr_node_ms = 0.0;
  DevBuf<int> b_doneround; DevBuf<double> d_tlimit; std::vector<double> round_elapsed; std::vector<int> h_doneround;   // per-plan solve times and limits
  DevBuf<unsigned char> d_prev_dec; DevBuf<double> d_prev_ub; DevBuf<unsigned long long> d_prev_uid; DevBuf<int> d_same;   // previous cycle (replan)
  DevBuf<unsigned long long> d_fp;                            // open-list fingerprints (frontier sharding)
  DevBuf<double> d_ubx;                                       // incumbent objectives exchanged between ranks (frontier sharding)
  double last_seconds = 0.0;
  bool timed_out = false;
  MiqpB200RunStats stats;
  DVec h_x;   // page-locked: D2H target of the solution vectors
  std::vector<double> h_viol, h_obj, h_bb, h_ub;
  std::vector<unsigned long long> h_stats;
  std::vector<int> h_done, h_overflow;
  std::vector<unsigned long long> h_incuid;
  std::vector<double> h_z;                                     // compact results: incumbent trajectories
  int single_maxN = 2;
  size_t pool_budget = 0;
  // solution pool: capacity requested for the next upload, device storage, fetch scratch (pool_* of BnbState)
  int solution_pool = 0;
  DevBuf<double> sp_z; DevBuf<unsigned char> sp_dec; DevBuf<PoolRec> sp_rec; DevBuf<int> sp_cnt;
  DevBuf<DevProb> sp_probs; DevBuf<int> sp_idx; DevBuf<double> sp_x, sp_zs, sp_obj, sp_viol;
  DevBuf<unsigned char> sp_export, sp_gathered;   // miqp_b200_pool_export's buffer; device copy of a merge input from elsewhere
  // streaming runs (miqp_b200_batch_run_streaming): callback (null outside such a run), delivered flags, harvest list, records
  // (device staging and page-locked host copy), records copied but not yet delivered, records held for the end of the run
  MiqpB200PlanDone on_done = nullptr; void *on_done_user = nullptr;
  DevBuf<int> hv_delivered, hv_list; DevBuf<double> hv_rec;
  DVec h_hvrec;
  std::vector<double> hv_held;
  cudaEvent_t ev_hv = nullptr;
  long hv_stride = 0;
  int hv_pending = 0, hv_bound = 0, hv_total = 0;
};

namespace {

int fail(MiqpB200Solver *s, int code, const std::string &msg) {
  if (s) s->err = msg;
  return code;
}

void upload_packed(MiqpB200Solver *s) {
  Packed &pk = s->pk;
  const int count = (int)pk.probs.size();
  s->d_probs.ensure(count);
  s->d_dblob.ensure(std::max<size_t>(pk.dblob.size() + (size_t)pk.dderived, 1));   // inputs of all plans, then the device-filled tables
  s->d_iblob.ensure(std::max<size_t>(pk.iblob.size() + (size_t)pk.iderived, 1));
  CK(cudaMemcpyAsync(s->d_probs.p, pk.probs.data(), sizeof(DevProb) * count, cudaMemcpyHostToDevice, s->stream));
  CK(cudaMemcpyAsync(s->d_dblob.p, pk.dblob.data(), sizeof(double) * pk.dblob.size(), cudaMemcpyHostToDevice, s->stream));
  CK(cudaMemcpyAsync(s->d_iblob.p, pk.iblob.data(), sizeof(int) * pk.iblob.size(), cudaMemcpyHostToDevice, s->stream));
  s->stats.h2d_bytes = (long)(sizeof(DevProb) * count + sizeof(double) * pk.dblob.size() + sizeof(int) * pk.iblob.size());
  launch_prepare_tables(s->d_probs.p, s->d_dblob.p, s->d_iblob.p, count, s->stream);
  CK(cudaGetLastError());
}

void pack_batch(MiqpB200Solver *s, const MiqpB200Problem *problems, int count) {
  Packed &pk = s->pk;
  pk.reset();   // keeps the page-locked capacity of the last batch
  s->time_limits.clear();
  for (int k = 0; k < count; ++k) s->time_limits.push_back(problems[k].time_limit);
  const int hw = (int)std::thread::hardware_concurrency();
  int cap = 8;   // packing threads; MIQP_PACK_THREADS lowers it when several processes / solver instances share the host cores
  if (const char *e = std::getenv("MIQP_PACK_THREADS")) cap = std::max(1, std::min(8, atoi(e)));
  const int nthr = std::max(1, std::min(std::min(cap, hw > 0 ? hw : 1), count / 128));
  if (nthr == 1) {
    for (int k = 0; k < count; ++k) {
      std::string v = validate(problems[k]);
      if (!v.empty()) throw std::invalid_argument("plan " + std::to_string(k) + ": " + v);
      pack_one(problems[k], pk);
    }
    for (DevProb &p : pk.probs) hostpack::place_plan(p, 0, 0, (long)pk.dblob.size(), (long)pk.iblob.size(), 0, 0, 0);
    return;
  }
  // large batches: workers pack contiguous shares into local blobs, which are then moved into the staging blobs
  std::vector<hostpack::PackedLocal> &part = s->pack_parts;   // kept between calls: no fresh pages to fault in
  part.resize(nthr);
  for (hostpack::PackedLocal &q : part) q.reset();
  std::vector<std::string> errs(nthr);
  {
    std::vector<std::thread> th;
    for (int t = 0; t < nthr; ++t)
      th.emplace_back([&, t]() {
        const int k0 = (int)((long)count * t / nthr), k1 = (int)((long)count * (t + 1) / nthr);
        for (int k = k0; k < k1; ++k) {
          std::string v = validate(problems[k]);
          if (!v.empty()) { errs[t] = "plan " + std::to_string(k) + ": " + v; return; }
          pack_one(problems[k], part[t]);
        }
      });
    for (std::thread &t : th) t.join();
  }
  for (const std::string &e : errs) if (!e.empty()) throw std::invalid_argument(e);
  std::vector<long> dbase(nthr + 1, 0), ibase(nthr + 1, 0), rbase(nthr + 1, 0), zbase(nthr + 1, 0), cbase(nthr + 1, 0), ddbase(nthr + 1, 0), idbase(nthr + 1, 0);
  for (int t = 0; t < nthr; ++t) {
    dbase[t + 1] = dbase[t] + (long)part[t].dblob.size(); ibase[t + 1] = ibase[t] + (long)part[t].iblob.size();
    ddbase[t + 1] = ddbase[t] + part[t].dderived; idbase[t + 1] = idbase[t] + part[t].iderived;
    rbase[t + 1] = rbase[t] + part[t].total_rows; zbase[t + 1] = zbase[t] + part[t].total_nnz; cbase[t + 1] = cbase[t] + part[t].total_cols;
    pk.max_rows = std::max(pk.max_rows, part[t].max_rows); pk.maxN = std::max(pk.maxN, part[t].maxN);
    pk.max_ndec = std::max(pk.max_ndec, part[t].max_ndec); pk.max_kmax = std::max(pk.max_kmax, part[t].max_kmax);
    pk.max_z = std::max(pk.max_z, part[t].max_z); pk.maxC = std::max(pk.maxC, part[t].maxC);
  }
  pk.total_rows = rbase[nthr]; pk.total_nnz = zbase[nthr]; pk.total_cols = cbase[nthr];
  pk.dderived = ddbase[nthr]; pk.iderived = idbase[nthr];
  pk.dblob.resize((size_t)dbase[nthr]); pk.iblob.resize((size_t)ibase[nthr]); pk.probs.resize(count);
  {
    std::vector<std::thread> th;
    for (int t = 0; t < nthr; ++t)
      th.emplace_back([&, t]() {
        std::memcpy(pk.dblob.data() + dbase[t], part[t].dblob.data(), sizeof(double) * part[t].dblob.size());
        std::memcpy(pk.iblob.data() + ibase[t], part[t].iblob.data(), sizeof(int) * part[t].iblob.size());
        const int k0 = (int)((long)count * t / nthr);
        for (size_t j = 0; j < part[t].probs.size(); ++j) {
          DevProb p = part[t].probs[j];
          hostpack::place_plan(p, dbase[t], ibase[t], dbase[nthr] + ddbase[t], ibase[nthr] + idbase[t], rbase[t], zbase[t], cbase[t]);
          pk.probs[k0 + j] = p;
        }
      });
    for (std::thread &t : th) t.join();
  }
}

// Solve info of plan k from its device results: batch_fetch and the deliveries of a streaming run build it alike.
void plan_info(const MiqpB200Solver *s, int k, double ub, unsigned long long incuid, double bb, double obj, double viol, int done,
               int done_round, int overflow, unsigned long long nodes, unsigned long long iters, unsigned long long uncert,
               MiqpB200SolveInfo &in) {
  const DevProb &p = s->pk.probs[k];
  std::memset(&in, 0, sizeof in);
  // (a finite bound without an incumbent of its own: the objective came from another rank, frontier sharding)
  const bool have = std::isfinite(ub) && incuid != ~0ULL;
  // solve time of THIS plan: the host's clock at the end of the round after which it was finished (the batch's time for a
  // plan that was still searching when the batch stopped)
  const int dr = done_round;
  in.seconds = (done && dr >= 1 && (size_t)(dr - 1) < s->round_elapsed.size() && s->round_elapsed[dr - 1] > 0.0) ? s->round_elapsed[dr - 1] : s->last_seconds;
  in.nodes = (long)nodes; in.qp_iters = (long)iters; in.rounds = s->stats.rounds;
  in.best_bound = bb;
  in.uncertified = (long)uncert;
  in.pool_exhausted = overflow;
  if (have) {
    // every open or pruned node may lie above the incumbent: report min(bound, incumbent) like CPLEX's best bound
    if (in.best_bound > ub) in.best_bound = ub;
    in.status = MIQP_B200_SUCCESS;
    in.objective = obj;  // re-evaluated on the full vector by evaluate_kernel
    in.max_violation = viol;
    const double lb = std::min(bb, ub);
    in.gap = std::fabs(lb - ub) / (1e-10 + std::fabs(ub));
    in.proven = (in.gap <= p.gap_tol + 1e-15) ? 1 : 0;
  } else {
    // no incumbent: the reference reports FAILED_TIMEOUT only for the time-limit status
    in.status = ((s->timed_out && !done) || done == 2) ? MIQP_B200_FAILED_TIMEOUT : MIQP_B200_FAILED_NO_SOLUT;
    in.objective = NAN; in.gap = NAN; in.max_violation = NAN;
  }
}

// ---- streaming runs -------------------------------------------------------------------------------------------------------
// Harvest of a round (after select): the plans select has just marked finished are finished like bnb_finish does it, evaluated
// and packed into records; their number lands in ctrl[7], which the host reads with the round's ctrl copy.  all = 1 (end of the
// run, after bnb_finish, which skips the delivered plans): every plan not delivered yet is evaluated and packed.
void launch_harvest(MiqpB200Solver *s, int all, int max_n) {
  int *list = s->hv_list.p, *n = s->b_ctrl.p + 7;
  launch_bnb_harvest(s->st, all, list, n, s->d_viol.p, s->stream);
  if (!all)
    launch_bnb_harvest_finish(s->st, s->d_probs.p, s->d_dblob.p, s->d_iblob.p, list, n, max_n, s->d_x.p, s->d_bb.p, s->stream);
  launch_evaluate_list(s->d_probs.p, s->d_dblob.p, s->d_iblob.p, list, n, max_n, s->pk.max_rows, s->d_x.p, s->d_viol.p, s->d_obj.p, s->stream);
  launch_bnb_harvest_pack(s->st, s->d_probs.p, list, n, max_n, s->d_obj.p, s->d_viol.p, s->d_bb.p, s->hv_rec.p, s->hv_stride, s->stream);
}

// copy of n records to the host (stream-ordered before the next harvest overwrites the staging area)
void copy_records(MiqpB200Solver *s, int n) {
  CK(cudaMemcpyAsync(s->h_hvrec.data(), s->hv_rec.p, sizeof(double) * (size_t)n * s->hv_stride, cudaMemcpyDeviceToHost, s->stream));
  CK(cudaEventRecord(s->ev_hv, s->stream));
  s->hv_pending = n;
  s->hv_total += n;
}

void deliver_record(MiqpB200Solver *s, const double *rec, long rounds) {
  StreamRec r;
  std::memcpy(&r, rec, sizeof r);
  MiqpB200SolveInfo in;
  plan_info(s, r.k, r.ub, r.inc_uid, r.best_bound, r.objective, r.max_violation, r.done, r.done_round, r.overflow, r.nodes, r.iters,
            r.uncert, in);
  in.rounds = rounds;
  s->on_done(s->on_done_user, r.k, rec + STREAM_REC_HDR, &in);
}

// Callbacks of the copied records, in ascending plan order.  A plan that finished before the first round (its time limit was over
// when the run started) reports the batch's time as its solve time, known only at the end: it is held and delivered then.
void deliver_pending(MiqpB200Solver *s) {
  if (s->hv_pending == 0) return;
  CK(cudaEventSynchronize(s->ev_hv));
  for (int e = 0; e < s->hv_pending; ++e) {
    const double *rec = s->h_hvrec.data() + (size_t)e * s->hv_stride;
    StreamRec r;
    std::memcpy(&r, rec, sizeof r);
    if (r.done_round >= 1) deliver_record(s, rec, r.done_round);
    else s->hv_held.insert(s->hv_held.end(), rec, rec + s->hv_stride);
  }
  s->hv_pending = 0;
}

// end of the run: the held plans and the plans stopped with the batch, merged in ascending plan order
void deliver_final(MiqpB200Solver *s) {
  CK(cudaEventSynchronize(s->ev_hv));
  std::vector<const double *> recs;
  for (size_t o = 0; o < s->hv_held.size(); o += (size_t)s->hv_stride) recs.push_back(s->hv_held.data() + o);
  for (int e = 0; e < s->hv_pending; ++e) recs.push_back(s->h_hvrec.data() + (size_t)e * s->hv_stride);
  std::sort(recs.begin(), recs.end(), [](const double *a, const double *b) {
    StreamRec ra, rb;
    std::memcpy(&ra, a, sizeof ra); std::memcpy(&rb, b, sizeof rb);
    return ra.k < rb.k;
  });
  s->hv_pending = 0;
  for (const double *rec : recs) deliver_record(s, rec, s->stats.rounds);
  s->hv_held.clear();
}

// Select / solve rounds of the uploaded batch, starting from the current device state: until every plan is finished, the time
// limit or round cap is hit, or `max_rounds_now` rounds have run (< 0: no such cap).  Returns the number of unfinished plans.
int run_rounds(MiqpB200Solver *s, long max_rounds_now) {
  double tlim = 0.0;
  for (double t : s->time_limits) tlim = std::max(tlim, t);
  int ctrl[8] = {s->fr_ctrl0, 0, 1, 0, 0, 0, 0, 0};
  long done_now = 0;
  for (;;) {
    if (max_rounds_now >= 0 && done_now >= max_rounds_now) break;
    const long rounds = s->fr_rounds;
    const double el0 = std::chrono::duration<double>(std::chrono::steady_clock::now() - s->fr_t0).count();
    if ((size_t)rounds >= s->round_elapsed.size()) s->round_elapsed.resize(rounds + 64, 0.0);
    launch_bnb_select(s->st, s->d_probs.p, (int)rounds + 1, el0, s->stream);
    s->fr_launches += 2;
    if (s->on_done) { launch_harvest(s, 0, rounds == 0 ? s->st.count : s->hv_bound); s->fr_launches += 4; }
    CK(cudaEventRecord(s->evr0, s->stream));
    if (s->n_single > 0) {
      // fewer single-car nodes than wide teams fit (work count of the last round as the estimate): latency matters, not throughput;
      // more than the four-warp teams hold at once: two-warp teams, twice as many nodes in flight
      const int est = (rounds == 0) ? s->n_single : ctrl[0];
      const bool wide = s->wide_ctas > 0 && rounds > 0 && est > 0 && est <= s->wide_ctas;
      const bool narrow = !wide && s->narrow_ctas > 0 && est >= s->narrow_min;
      int rc = narrow ? launch_bnb_nodes(s->st, s->d_probs.p, s->d_dblob.p, s->d_iblob.p, s->smem_narrow, NODE_TEAM_WARPS_NARROW,
                                         s->narrow_ctas, s->single_maxN, s->narrow_np, (int)rounds + 1, s->stream)
                      : launch_bnb_nodes(s->st, s->d_probs.p, s->d_dblob.p, s->d_iblob.p, s->smem_per_warp,
                                         wide ? NODE_TEAM_WARPS_WIDE : s->warps_per_cta, wide ? s->wide_ctas : s->ctas, s->single_maxN,
                                         s->single_maxN + 7, (int)rounds + 1, s->stream);
      if (narrow) ++s->narrow_launches;
      if (rc != 0) throw std::runtime_error(std::string("node kernel launch failed: ") + cudaGetErrorString((cudaError_t)rc));
      ++s->fr_launches; ++s->fr_node_launches;
    }
    if (s->n_multi > 0) {
      int rc = launch_bnb_nodes_multi(s->st, s->d_probs.p, s->d_dblob.p, s->d_iblob.p, s->b_multi_ws.p, s->multi_ws_bytes,
                                      s->multi_use_smem, s->multi_threads, s->multi_ctas, (int)rounds + 1, s->stream);
      if (rc != 0) throw std::runtime_error(std::string("multi-car node kernel launch failed: ") + cudaGetErrorString((cudaError_t)rc));
      ++s->fr_launches; ++s->fr_node_launches;
    }
    CK(cudaEventRecord(s->evr1, s->stream));
    if (s->on_done) deliver_pending(s);   // the last round's plans, while this round's node kernels run
    ++s->fr_rounds; ++done_now;
    CK(cudaMemcpyAsync(ctrl, s->b_ctrl.p, sizeof ctrl, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    s->fr_ctrl0 = ctrl[0];
    if (s->on_done) {
      s->hv_bound = ctrl[2];   // only plans active in this round can finish in the next select
      if (ctrl[7] > 0) copy_records(s, ctrl[7]);
    }
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, s->evr0, s->evr1));
    s->fr_node_ms += ms;
    if (s->opt.verbose > 1) fprintf(stderr, "[miqp_b200] round %ld: work %d active %d err %d node kernel %.3f ms (narrow launches so far %ld)\n", s->fr_rounds, ctrl[0], ctrl[2], ctrl[3], ms, s->narrow_launches);
    if (ctrl[2] == 0) break;  // every plan finished
    const double el = std::chrono::duration<double>(std::chrono::steady_clock::now() - s->fr_t0).count();
    s->round_elapsed[rounds] = el;   // (rounds = index of the round that just ended, counted from 0)
    if (el > tlim) { s->timed_out = true; break; }
    if (s->opt.max_rounds > 0 && s->fr_rounds >= s->opt.max_rounds) { s->timed_out = true; break; }
  }
  return ctrl[2];
}

// Start of a search of the uploaded batch, for batch runs and the stepped search (miqp_b200_frontier_*) alike: fresh search
// state, the run's counters and its clocks.  A streaming run also clears its delivered flags.
void start_run(MiqpB200Solver *s) {
  const int count = s->st.count;
  s->fr_t0 = std::chrono::steady_clock::now();
  CK(cudaMemsetAsync(s->b_prof.p, 0, 256 * sizeof(unsigned long long), s->stream));
  if (s->st.susp_slot) CK(cudaMemsetAsync(s->st.susp_slot, 0xff, sizeof(int) * (size_t)count * s->st.cap, s->stream));
  if (s->on_done) {
    s->hv_stride = (STREAM_REC_HDR + (long)s->pk.maxC * s->pk.maxN * 8 + 1) & ~1L;   // records 16-byte aligned
    s->hv_delivered.ensure(count); s->hv_list.ensure(count); s->hv_rec.ensure((size_t)count * s->hv_stride);
    s->h_hvrec.resize((size_t)count * s->hv_stride);
    if (!s->ev_hv) CK(cudaEventCreateWithFlags(&s->ev_hv, cudaEventDisableTiming));
    CK(cudaMemsetAsync(s->hv_delivered.p, 0, sizeof(int) * count, s->stream));
    s->st.delivered = s->hv_delivered.p;
    s->hv_pending = 0; s->hv_total = 0; s->hv_held.clear();
  }
  CK(cudaEventRecord(s->ev0, s->stream));
  launch_bnb_init(s->st, s->d_probs.p, s->any_warm ? s->d_warm.p : nullptr, s->any_warm ? s->d_haswarm.p : nullptr, s->stream);
  s->fr_rounds = 0; s->fr_ctrl0 = 0;
  s->fr_launches = 1; s->fr_node_launches = 0; s->fr_node_ms = 0.0;
  s->timed_out = false; s->ran = false;
}

// End of a search: final solution vectors and their evaluation, then the run's device time and statistics.  A streaming run
// delivers the plans of its last round first, and the plans still searching when the batch stopped last (same evaluate code).
void finish_run(MiqpB200Solver *s, float *device_ms) {
  const bool streaming = s->on_done != nullptr;
  const int count = s->st.count;
  if (streaming) deliver_pending(s);
  launch_bnb_finish(s->st, s->d_probs.p, s->d_dblob.p, s->d_iblob.p, s->d_x.p, s->d_bb.p, s->stream);
  if (!streaming) {
    CK(cudaMemsetAsync(s->d_viol.p, 0, sizeof(double) * count, s->stream));
    launch_evaluate(s->d_probs.p, s->d_dblob.p, s->d_iblob.p, count, s->pk.max_rows, s->d_x.p, s->d_viol.p, s->d_obj.p, s->stream);
  } else {   // exactly the plans not delivered yet
    const int left = count - s->hv_total;
    launch_harvest(s, 1, left);
    s->fr_launches += 2;
    if (left > 0) copy_records(s, left);
  }
  s->fr_launches += 2;
  CK(cudaGetLastError());
  CK(cudaEventRecord(s->ev1, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  float total_ms = 0.f;
  CK(cudaEventElapsedTime(&total_ms, s->ev0, s->ev1));
  if (device_ms) *device_ms = total_ms;
  s->last_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - s->fr_t0).count();
  s->stats.launches = s->fr_launches; s->stats.node_kernel_launches = s->fr_node_launches; s->stats.rounds = s->fr_rounds;
  s->stats.node_kernel_ms = s->fr_node_ms; s->stats.total_ms = total_ms;
  s->ran = true;
  if (streaming) deliver_final(s);
}

void setup_bnb(MiqpB200Solver *s) {
  Packed &pk = s->pk;
  const int count = (int)pk.probs.size();
  BnbState &st = s->st;
  st.count = count;
  st.ndec_stride = pk.max_ndec;
  st.zstride = pk.max_z;
  st.kmax = pk.max_kmax;
  st.npad = ((pk.maxN + 31) / 32) * 32;
  // node kernel geometry: warp-per-node kernel for single-car plans, CTA-per-node kernel otherwise
  int maxN1 = 0, minN1 = 1 << 30, kmax1 = 0, maxCm = 0;
  s->n_single = 0; s->n_multi = 0; s->multi_ws_bytes = 0;
  const char *fm = std::getenv("MIQP_B200_FORCE_MULTI");   // test hook: run single-car plans through the CTA-per-node kernel
  st.force_multi = (fm && fm[0] == '1') ? 1 : 0;
  for (const DevProb &p : pk.probs) {
    if (p.C == 1 && !st.force_multi) { ++s->n_single; maxN1 = std::max(maxN1, p.N); minN1 = std::min(minN1, p.N); kmax1 = std::max(kmax1, p.kmax); }
    else {
      ++s->n_multi; maxCm = std::max(maxCm, p.C);
      s->multi_ws_bytes = std::max(s->multi_ws_bytes, multi_workspace_bytes(p.C, p.N, p.P, p.kmax, st.ndec_stride));
    }
  }
  st.kmax = std::max(kmax1, 1);
  s->single_maxN = std::max(maxN1, 2);
  st.nwarps = 0; s->ctas = 0; s->multi_ctas = 0;
  if (s->n_single > 0) {
    s->smem_per_warp = node_kernel_smem_per_warp(s->single_maxN, st.kmax, st.ndec_stride);   // per node (one team)
    s->warps_per_cta = NODE_TEAM_WARPS;
    const int per_sm = node_kernel_max_ctas(s->smem_per_warp, s->warps_per_cta * 32);
    if (per_sm <= 0) throw std::runtime_error("node kernel does not fit in shared memory for this horizon");
    s->ctas = per_sm * s->num_sms;
    s->wide_ctas = 0;
    if (!getenv("MIQP_NO_WIDE_TEAM")) {
      const int wide_per_sm = node_kernel_max_ctas(s->smem_per_warp, NODE_TEAM_WARPS_WIDE * 32);
      if (wide_per_sm > 0) s->wide_ctas = wide_per_sm * s->num_sms;
    }
    // two-warp teams (four per SM) for rounds with many nodes; only when every single-car plan has the same horizon (the
    // shared-memory layout then uses the row stride of that team size)
    s->narrow_ctas = 0; s->narrow_launches = 0;
    if (!getenv("MIQP_NO_NARROW_TEAM") && minN1 == maxN1) {
      s->narrow_np = node_kernel_narrow_np(maxN1);
      s->smem_narrow = node_kernel_smem_narrow(maxN1, st.kmax, st.ndec_stride);
      const int narrow_per_sm = node_kernel_max_ctas(s->smem_narrow, NODE_TEAM_WARPS_NARROW * 32);
      if (narrow_per_sm > per_sm) s->narrow_ctas = narrow_per_sm * s->num_sms;   // only if more nodes are in flight than with four-warp teams
      s->narrow_min = 2 * s->ctas;   // between one and two waves of four-warp teams the two variants take the same time; the wider team has the lower latency
      if (const char *e = getenv("MIQP_NARROW_MIN")) s->narrow_min = atoi(e);
    }
    st.nwarps += 2 * s->num_sms;   // the round-width rules are tuned for two teams per SM, whatever the launch uses
  }
  if (s->n_multi > 0) {
    s->multi_threads = (maxCm <= 2) ? 64 : 128;
    int per_sm = (s->multi_ws_bytes <= 220 * 1024) ? multi_kernel_max_ctas((int)s->multi_ws_bytes, s->multi_threads) : 0;
    if (per_sm > 0) { s->multi_use_smem = 1; }
    else {  // working set of a node does not fit in shared memory: per-CTA slice of HBM (L2 resident)
      s->multi_use_smem = 0;
      per_sm = std::min(4, std::max(1, multi_kernel_max_ctas(0, s->multi_threads)));
    }
    s->multi_ctas = per_sm * s->num_sms;
    if (!s->multi_use_smem) s->b_multi_ws.ensure((size_t)s->multi_ctas * (size_t)s->multi_ws_bytes / 8 + 16);
    st.nwarps += s->multi_ctas;
  }
  // nodes per plan per round.  Base count: enough to fill the resident warps once (every extra node
  // per round is speculative: 37 -> 45 -> 53 nodes per config-2 plan at 1 / 3 / 5); one dive head
  // per plan until an incumbent exists; up to KS when few plans are still active.
  int K = s->opt.nodes_per_round;
  if (K <= 0) { K = (st.nwarps + count - 1) / count; if (K < 1) K = 1; if (K > 64) K = 64; }
  st.sel_base = K;
  st.sel_dive = std::max(1, std::min(8, st.nwarps / std::max(count, 1)));   // several dive heads only when warps would idle
  st.dive_fill = 2;   // A/B on 2048 config-2 plans (profiles/r1i, r1k): one dive head 347 ms / 120 rounds; widened dive 143 ms / 53 rounds
  if (const char *e = getenv("MIQP_DIVE_FILL")) st.dive_fill = atoi(e);
  st.dive_patience = 14; st.dive_growth = 8;   // profiles/r1k: batch 1024 139 -> 80 ms, batch 2048 unchanged (144 ms, 53 -> 38 rounds)
  if (const char *e = getenv("MIQP_DIVE_PATIENCE")) st.dive_patience = atoi(e);
  if (const char *e = getenv("MIQP_DIVE_GROWTH")) st.dive_growth = atoi(e);
  st.multi_heur = 1;
  if (const char *e = getenv("MIQP_MULTI_HEUR")) st.multi_heur = atoi(e);
  int kscap = 64;
  // a few multi-car plans alone on the GPU (config 5: ONE joint plan): let a plan take as many nodes per round as CTAs are resident
  if (s->n_single == 0 && s->n_multi > 0) kscap = std::max(64, std::min(1024, st.nwarps / std::max(count, 1)));
  if (const char *e = getenv("MIQP_KS")) kscap = std::max(1, atoi(e));
  int KS = std::max(K, std::min(kscap, std::max(1, st.nwarps)));
  st.sel_per_plan = KS;
  // pool capacity per plan
  int cap = s->opt.pool_capacity;
  // warm start of the children from the parent's relaxed optimum (single-car nodes): N x 8 doubles per node
  st.warm_mu = 10.0; st.zp_stride = 0;   // profiles/r1k: with parked relaxations 84.2 -> 76.9 ms (2048 plans), 8.6 -> 7.7 iterations per node
  st.tau_k = 1.0;   // profiles/r1k: 9.45 -> 8.6 interior-point iterations per node
  if (const char *e = getenv("MIQP_TAU_K")) st.tau_k = atof(e);
  if (const char *e = getenv("MIQP_WARM_MU")) st.warm_mu = atof(e);
  if (st.warm_mu > 0.0 && s->n_single > 0) st.zp_stride = s->single_maxN * 8;
  if (cap <= 0) {
    const size_t node_bytes = (size_t)st.ndec_stride + 48 + (size_t)8 * st.zp_stride;
    // pool budget: a quarter of the free HBM, at most 24 GiB (B200: 180 GB per GPU; several solver instances share a GPU when
    // batches are pipelined: capi.PipelinedSolver)
    if (s->pool_budget == 0) {   // asked once per solver: cudaMemGetInfo costs about a millisecond
      size_t free_b = 0, total_b = 0;
      s->pool_budget = (size_t)8 << 30;
      if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) s->pool_budget = std::min<size_t>(free_b / 4, (size_t)24 << 30);
    }
    const size_t budget = s->pool_budget;
    size_t c = budget / (node_bytes * (size_t)count);
    if (c > (1u << 20)) c = 1u << 20;
    if (c < 256) c = 256;
    cap = (int)c;
  }
  if (cap < 4 * KS + 64) cap = 4 * KS + 64;
  st.cap = cap;
  st.work_cap = count * KS;
  const size_t nodes = (size_t)count * cap;
  s->b_dec.ensure(nodes * st.ndec_stride); st.dec = s->b_dec.p;
  s->b_bound.ensure(nodes); st.bound = s->b_bound.p;
  // parked relaxations (single-car nodes): iteration budget per round, two state pools written alternately
  st.susp_budget = 8;   // profiles/r1k: cold starts 10 was best (129 -> 86 ms); with the warm start 6 / 7 / 8 / 10 / 12: 88 / 83 / 69 / 77 / 88 ms per 2048 plans
  if (const char *e = getenv("MIQP_SUSP_BUDGET")) st.susp_budget = atoi(e);
  st.susp_slot = nullptr; st.susp_cnt = nullptr; st.susp_pool[0] = st.susp_pool[1] = nullptr; st.susp_slots = 0; st.susp_stride = 0;
  if (st.susp_budget > 0 && s->n_single > 0) {
    const int np = s->single_maxN + 7;
    st.susp_stride = (8 + (long)s->single_maxN * 35 + 1 + 2L * (st.kmax + 1) * np + 1) & ~1L;   // SUSP_HDR + V + (s, lambda) records, 16-byte aligned
    st.susp_slots = std::min(st.work_cap, 4096);
    s->b_susp0.ensure((size_t)st.susp_slots * st.susp_stride); s->b_susp1.ensure((size_t)st.susp_slots * st.susp_stride);
    st.susp_pool[0] = s->b_susp0.p; st.susp_pool[1] = s->b_susp1.p;
    s->b_suspslot.ensure(nodes); st.susp_slot = s->b_suspslot.p;
    s->b_suspcnt.ensure(1); st.susp_cnt = s->b_suspcnt.p;
  }
  st.zpool = nullptr;
  if (st.zp_stride > 0) { s->b_zpool.ensure(nodes * (size_t)st.zp_stride); st.zpool = s->b_zpool.p; }
  s->b_meta.ensure(nodes); st.meta = s->b_meta.p;
  s->b_uid.ensure(nodes); st.uid = s->b_uid.p;
  s->b_open.ensure(nodes); st.open_idx = s->b_open.p;
  s->b_free.ensure(nodes); st.free_stack = s->b_free.p;
  s->b_keybuf.ensure(nodes); st.keybuf = s->b_keybuf.p;
  s->b_opencnt.ensure(count); st.open_cnt = s->b_opencnt.p;
  s->b_freecnt.ensure(count); st.free_cnt = s->b_freecnt.p;
  s->b_sel.ensure((size_t)count * KS); st.sel_idx = s->b_sel.p;
  s->b_selcnt.ensure(count); st.sel_cnt = s->b_selcnt.p;
  s->b_ub.ensure(count); st.ub = s->b_ub.p;
  s->b_cutoff.ensure(count); st.cutoff = s->b_cutoff.p;
  s->b_pruned.ensure(count); st.pruned_lb = s->b_pruned.p;
  s->b_done.ensure(count); st.done = s->b_done.p;
  s->b_doneround.ensure(count); st.done_round = s->b_doneround.p;
  s->d_tlimit.ensure(count); st.tlimit = s->d_tlimit.p;
  CK(cudaMemcpyAsync(s->d_tlimit.p, s->time_limits.data(), sizeof(double) * count, cudaMemcpyHostToDevice, s->stream));
  s->b_lock.ensure(count); st.lock = s->b_lock.p;
  s->b_incz.ensure((size_t)count * st.zstride); st.inc_z = s->b_incz.p;
  s->b_incdec.ensure((size_t)count * st.ndec_stride); st.inc_dec = s->b_incdec.p;
  s->b_incuid.ensure(count); st.inc_uid = s->b_incuid.p;
  s->b_stats.ensure((size_t)4 * count);
  st.stat_nodes = s->b_stats.p; st.stat_iters = s->b_stats.p + count; st.stat_rows = s->b_stats.p + 2 * count; st.stat_uncert = s->b_stats.p + 3 * count;
  s->b_overflow.ensure(count); st.overflow = s->b_overflow.p;
  s->b_work.ensure(st.work_cap); st.work = s->b_work.p;
  s->b_work2.ensure(st.work_cap); st.work2 = s->b_work2.p;
  s->b_ctrl.ensure(8);
  s->b_prof.ensure(256); st.prof = s->b_prof.p;
  s->b_dbg.ensure((size_t)(1024 + 8) * 512); st.dbg = s->b_dbg.p;
  st.work_cnt = s->b_ctrl.p; st.work_next = s->b_ctrl.p + 1; st.active = s->b_ctrl.p + 2; st.err = s->b_ctrl.p + 3;
  st.work_cnt2 = s->b_ctrl.p + 4; st.work_next2 = s->b_ctrl.p + 5; st.active_prev = s->b_ctrl.p + 6;
  s->d_x.ensure(std::max<long>(pk.total_cols, 1));
  s->d_viol.ensure(count); s->d_obj.ensure(count); s->d_bb.ensure(count);
  // solution pool: storage only when it is on (config 2: about 3.2 kB per entry)
  st.pool_cap = s->solution_pool;
  st.pool_z = nullptr; st.pool_dec = nullptr; st.pool_rec = nullptr; st.pool_cnt = nullptr;
  if (st.pool_cap > 0) {
    const size_t entries = (size_t)count * st.pool_cap;
    s->sp_z.ensure(entries * st.zstride); st.pool_z = s->sp_z.p;
    s->sp_dec.ensure(entries * st.ndec_stride); st.pool_dec = s->sp_dec.p;
    s->sp_rec.ensure(entries); st.pool_rec = s->sp_rec.p;
    s->sp_cnt.ensure(count); st.pool_cnt = s->sp_cnt.p;
  }
}

}  // namespace

// ---- pool export layout (miqp_b200_pool_export / miqp_b200_pool_merge) ----------------------------------------------------
namespace {
constexpr unsigned POOL_EXPORT_MAGIC = 0x4c4f4f50u;   // "POOL"
constexpr unsigned POOL_EXPORT_VERSION = 1;
struct PoolExportHeader {   // first 64 bytes of an export
  unsigned magic, version;
  int count, cap, zstride, ndec_stride;
  unsigned long long shape_hash;   // FNV-1a over (C, N, R, O, L, E, ncols) of every plan
  unsigned char pad[32];
};
static_assert(sizeof(PoolExportHeader) == 64, "export header size");

long align16(long b) { return (b + 15) & ~15L; }

PoolExportLayout export_layout(const BnbState &st) {
  PoolExportLayout l;
  const long entries = (long)st.count * st.pool_cap;
  l.off_cnt = sizeof(PoolExportHeader);
  l.off_rec = align16(l.off_cnt + (long)sizeof(int) * st.count);
  l.off_dec = align16(l.off_rec + (long)sizeof(PoolRec) * entries);
  l.off_z = align16(l.off_dec + entries * st.ndec_stride);
  l.bytes = align16(l.off_z + (long)sizeof(double) * entries * st.zstride);
  return l;
}

PoolExportHeader export_header(const MiqpB200Solver *s) {
  PoolExportHeader h;
  std::memset(&h, 0, sizeof h);
  h.magic = POOL_EXPORT_MAGIC; h.version = POOL_EXPORT_VERSION;
  h.count = s->st.count; h.cap = s->st.pool_cap; h.zstride = s->st.zstride; h.ndec_stride = s->st.ndec_stride;
  unsigned long long f = 0xcbf29ce484222325ULL;
  for (const DevProb &p : s->pk.probs)
    for (int v : {p.C, p.N, p.R, p.O, p.L, p.E, p.ncols}) { f ^= (unsigned)v; f *= 0x100000001b3ULL; }
  h.shape_hash = f;
  return h;
}
}  // namespace

extern "C" {

const char *miqp_b200_version(void) { return "planner-miqp_b200 0.1 (sm_100a)"; }

void miqp_b200_default_options(MiqpB200Options *opt) {
  if (!opt) return;
  opt->device = 0; opt->nodes_per_round = 0; opt->pool_capacity = 0; opt->max_rounds = 0; opt->verbose = 0;
}

int miqp_b200_create(const MiqpB200Options *opt, MiqpB200Solver **out) {
  if (!out) return MIQP_B200_ERR_ARG;
  *out = nullptr;
  MiqpB200Solver *s = new MiqpB200Solver();
  if (opt) s->opt = *opt; else miqp_b200_default_options(&s->opt);
  std::memset(&s->stats, 0, sizeof s->stats);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= s->opt.device) {
    fprintf(stderr, "miqp_b200: no usable CUDA device (%s); this backend has no CPU fallback\n",
            e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range");
    delete s;
    return MIQP_B200_ERR_CUDA;
  }
  try {
    CK(cudaSetDevice(s->opt.device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, s->opt.device));
    s->num_sms = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&s->ev0)); CK(cudaEventCreate(&s->ev1));
    CK(cudaEventCreate(&s->evr0)); CK(cudaEventCreate(&s->evr1));
    CK(cudaEventCreate(&s->mark[0])); CK(cudaEventCreate(&s->mark[1]));
  } catch (const std::exception &ex) {
    fprintf(stderr, "miqp_b200: %s\n", ex.what());
    delete s;
    return MIQP_B200_ERR_CUDA;
  }
  *out = s;
  return MIQP_B200_OK;
}

void miqp_b200_destroy(MiqpB200Solver *s) {
  if (!s) return;
  cudaSetDevice(s->opt.device);
  s->d_probs.release(); s->d_dblob.release(); s->d_iblob.release(); s->d_x.release(); s->d_viol.release();
  s->d_obj.release(); s->d_bb.release(); s->d_warm.release(); s->d_haswarm.release();
  s->a_rowptr.release(); s->a_cols.release(); s->a_vals.release(); s->a_lo.release(); s->a_hi.release(); s->a_cnt.release();
  s->b_dec.release(); s->b_incdec.release(); s->b_bound.release(); s->b_ub.release(); s->b_cutoff.release();
  s->b_pruned.release(); s->b_incz.release(); s->b_meta.release(); s->b_work.release();
  s->b_uid.release(); s->b_keybuf.release(); s->b_incuid.release(); s->b_stats.release(); s->b_open.release();
  s->b_opencnt.release(); s->b_free.release(); s->b_freecnt.release(); s->b_sel.release(); s->b_selcnt.release();
  s->sp_z.release(); s->sp_dec.release(); s->sp_rec.release(); s->sp_cnt.release(); s->sp_export.release(); s->sp_gathered.release();
  s->b_zpool.release(); s->b_susp0.release(); s->b_susp1.release(); s->b_suspslot.release(); s->b_suspcnt.release(); s->b_done.release(); s->b_overflow.release(); s->b_lock.release(); s->b_ctrl.release(); s->b_multi_ws.release(); s->b_work2.release();
  if (s->ev0) cudaEventDestroy(s->ev0);
  if (s->ev1) cudaEventDestroy(s->ev1);
  if (s->evr0) cudaEventDestroy(s->evr0);
  if (s->mark[0]) cudaEventDestroy(s->mark[0]);
  if (s->mark[1]) cudaEventDestroy(s->mark[1]);
  if (s->evr1) cudaEventDestroy(s->evr1);
  if (s->ev_hv) cudaEventDestroy(s->ev_hv);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;
}

const char *miqp_b200_last_error(const MiqpB200Solver *s) { return s ? s->err.c_str() : "null solver"; }

int miqp_b200_layout(const MiqpB200Problem *p, MiqpB200Layout *out) {
  if (!p || !out) return MIQP_B200_ERR_ARG;
  layout_of(*p, *out);
  return MIQP_B200_OK;
}

int miqp_b200_assemble(MiqpB200Solver *s, const MiqpB200Problem *p, long *rowptr, int *cols, double *vals,
                       double *lo, double *hi) {
  MiqpB200Sizes sz;
  if (!s || !p) return MIQP_B200_ERR_ARG;
  try {
    CK(cudaSetDevice(s->opt.device));
    pack_batch(s, p, 1);
    s->uploaded = false;
    upload_packed(s);
    const long rows = s->pk.total_rows, nnz = s->pk.total_nnz;
    s->a_rowptr.ensure(rows + 1); s->a_cols.ensure(std::max<long>(nnz, 1)); s->a_vals.ensure(std::max<long>(nnz, 1));
    s->a_lo.ensure(rows + 1); s->a_hi.ensure(rows + 1); s->a_cnt.ensure(1);
    CK(cudaMemsetAsync(s->a_cnt.p, 0, sizeof(unsigned long long), s->stream));
    launch_assemble_rows(s->d_probs.p, s->d_dblob.p, s->d_iblob.p, 1, s->pk.max_rows, s->a_rowptr.p, s->a_cols.p, s->a_vals.p,
                         s->a_lo.p, s->a_hi.p, s->a_cnt.p, s->stream);
    CK(cudaGetLastError());
    if (rowptr) CK(cudaMemcpyAsync(rowptr, s->a_rowptr.p, sizeof(long) * (rows + 1), cudaMemcpyDeviceToHost, s->stream));
    if (cols) CK(cudaMemcpyAsync(cols, s->a_cols.p, sizeof(int) * nnz, cudaMemcpyDeviceToHost, s->stream));
    if (vals) CK(cudaMemcpyAsync(vals, s->a_vals.p, sizeof(double) * nnz, cudaMemcpyDeviceToHost, s->stream));
    if (lo) CK(cudaMemcpyAsync(lo, s->a_lo.p, sizeof(double) * rows, cudaMemcpyDeviceToHost, s->stream));
    if (hi) CK(cudaMemcpyAsync(hi, s->a_hi.p, sizeof(double) * rows, cudaMemcpyDeviceToHost, s->stream));
    unsigned long long cnt = 0;
    CK(cudaMemcpyAsync(&cnt, s->a_cnt.p, sizeof cnt, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    s->stats.launches += 2;
    sz.nnz = (long)cnt;
    s->h_stats.assign(1, cnt);
  } catch (const std::invalid_argument &ex) {
    return fail(s, MIQP_B200_ERR_ARG, ex.what());
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

int miqp_b200_assemble_batch(MiqpB200Solver *s, const MiqpB200Problem *problems, int count, int repeats, float *device_ms,
                             long *rows_out, long *nnz_out) {
  if (!s || !problems || count <= 0) return MIQP_B200_ERR_ARG;
  try {
    CK(cudaSetDevice(s->opt.device));
    pack_batch(s, problems, count);
    s->uploaded = false;
    upload_packed(s);
    const long rows = s->pk.total_rows, nnz = s->pk.total_nnz;
    // every plan owns nrows + 1 row pointers and its own non-zero counter (formulation.cu:assemble_rows_kernel)
    s->a_rowptr.ensure(rows + count); s->a_cols.ensure(std::max<long>(nnz, 1)); s->a_vals.ensure(std::max<long>(nnz, 1));
    s->a_lo.ensure(rows + count); s->a_hi.ensure(rows + count); s->a_cnt.ensure(count);
    CK(cudaMemsetAsync(s->a_cnt.p, 0, sizeof(unsigned long long) * count, s->stream));
    const int reps = std::max(repeats, 1);
    // one untimed pass (first touch of the output pages), then `reps` timed ones
    launch_assemble_rows(s->d_probs.p, s->d_dblob.p, s->d_iblob.p, count, s->pk.max_rows, s->a_rowptr.p, s->a_cols.p, s->a_vals.p,
                         s->a_lo.p, s->a_hi.p, s->a_cnt.p, s->stream);
    CK(cudaEventRecord(s->ev0, s->stream));
    for (int r = 0; r < reps; ++r)
      launch_assemble_rows(s->d_probs.p, s->d_dblob.p, s->d_iblob.p, count, s->pk.max_rows, s->a_rowptr.p, s->a_cols.p, s->a_vals.p,
                           s->a_lo.p, s->a_hi.p, s->a_cnt.p, s->stream);
    CK(cudaEventRecord(s->ev1, s->stream));
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s->stream));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    if (device_ms) *device_ms = ms / reps;
    if (rows_out) *rows_out = rows;
    if (nnz_out) *nnz_out = nnz;
    s->stats.launches += 1 + reps;
  } catch (const std::invalid_argument &ex) {
    return fail(s, MIQP_B200_ERR_ARG, ex.what());
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

int miqp_b200_sizes(MiqpB200Solver *s, const MiqpB200Problem *p, MiqpB200Sizes *out) {
  if (!s || !p || !out) return MIQP_B200_ERR_ARG;
  int rc = miqp_b200_assemble(s, p, nullptr, nullptr, nullptr, nullptr, nullptr);
  if (rc != MIQP_B200_OK) return rc;
  MiqpB200Layout l; layout_of(*p, l);
  out->ncols = l.ncols;
  out->nbin = (l.base_so - l.base_nwe) + (l.base_sv - l.base_c2c);
  out->ncont = l.ncols - out->nbin;
  out->nrows = s->pk.total_rows; out->nnz_struct = s->pk.total_nnz;
  out->nnz = (long)s->h_stats[0];
  return MIQP_B200_OK;
}

int miqp_b200_evaluate(MiqpB200Solver *s, const MiqpB200Problem *p, const double *x, double *objective,
                       double *max_violation) {
  if (!s || !p || !x) return MIQP_B200_ERR_ARG;
  try {
    CK(cudaSetDevice(s->opt.device));
    pack_batch(s, p, 1);
    s->uploaded = false;
    upload_packed(s);
    s->d_x.ensure(s->pk.total_cols); s->d_viol.ensure(1); s->d_obj.ensure(1);
    CK(cudaMemcpyAsync(s->d_x.p, x, sizeof(double) * s->pk.total_cols, cudaMemcpyHostToDevice, s->stream));
    CK(cudaMemsetAsync(s->d_viol.p, 0, sizeof(double), s->stream));
    launch_evaluate(s->d_probs.p, s->d_dblob.p, s->d_iblob.p, 1, s->pk.max_rows, s->d_x.p, s->d_viol.p, s->d_obj.p, s->stream);
    CK(cudaGetLastError());
    double v = 0, o = 0;
    CK(cudaMemcpyAsync(&v, s->d_viol.p, sizeof v, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(&o, s->d_obj.p, sizeof o, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    s->stats.launches += 2;
    if (objective) *objective = o;
    if (max_violation) *max_violation = v;
  } catch (const std::invalid_argument &ex) {
    return fail(s, MIQP_B200_ERR_ARG, ex.what());
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

int miqp_b200_batch_upload(MiqpB200Solver *s, const MiqpB200Problem *problems, int count, const double *const *warm) {
  if (!s || !problems || count <= 0) return MIQP_B200_ERR_ARG;
  try {
    CK(cudaSetDevice(s->opt.device));
    s->uploaded = false; s->ran = false;
    const auto tp0 = std::chrono::steady_clock::now();
    pack_batch(s, problems, count);
    const auto tp1 = std::chrono::steady_clock::now();
    upload_packed(s);
    setup_bnb(s);
    // MIP starts
    s->any_warm = false;
    s->h_haswarm.assign(count, 0);
    s->h_warm.assign((size_t)count * s->st.ndec_stride, UNDEC);
    if (warm)
      for (int k = 0; k < count; ++k)
        if (warm[k]) {
          std::vector<int> dummy;
          decisions_from_solution(problems[k], s->pk.probs[k], dummy, warm[k], s->h_warm.data() + (size_t)k * s->st.ndec_stride);
          s->h_haswarm[k] = 1; s->any_warm = true;
        }
    if (s->any_warm) {
      s->d_warm.ensure(s->h_warm.size()); s->d_haswarm.ensure(count);
      CK(cudaMemcpyAsync(s->d_warm.p, s->h_warm.data(), s->h_warm.size(), cudaMemcpyHostToDevice, s->stream));
      CK(cudaMemcpyAsync(s->d_haswarm.p, s->h_haswarm.data(), sizeof(int) * count, cudaMemcpyHostToDevice, s->stream));
      s->stats.h2d_bytes += (long)(s->h_warm.size() + sizeof(int) * count);
    }
    CK(cudaStreamSynchronize(s->stream));
    s->stats.pack_ms = std::chrono::duration<double, std::milli>(tp1 - tp0).count();
    s->stats.upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tp1).count();
    s->uploaded = true;
  } catch (const std::invalid_argument &ex) {
    return fail(s, MIQP_B200_ERR_ARG, ex.what());
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

// Receding-horizon replanning without a host round trip of the solutions: the MIP start of every plan is the incumbent of the
// previous batch on this solver (same plan order, same shapes), shifted by one step on the device (bnb_shift_warm_kernel).
int miqp_b200_batch_upload_replan(MiqpB200Solver *s, const MiqpB200Problem *problems, int count) {
  if (!s || !problems || count <= 0) return MIQP_B200_ERR_ARG;
  if (!s->ran) return fail(s, MIQP_B200_ERR_ARG, "batch_upload_replan needs the results of a previous batch_run on this solver");
  if (count != s->st.count) return fail(s, MIQP_B200_ERR_ARG, "batch_upload_replan: the batch must hold the same plans as the previous one");
  try {
    CK(cudaSetDevice(s->opt.device));
    // the previous cycle's incumbents, before the buffers are reused
    const int prev_stride = s->st.ndec_stride;
    s->d_prev_dec.ensure((size_t)count * prev_stride); s->d_prev_ub.ensure(count); s->d_prev_uid.ensure(count); s->d_same.ensure(count);
    CK(cudaMemcpyAsync(s->d_prev_dec.p, s->st.inc_dec, (size_t)count * prev_stride, cudaMemcpyDeviceToDevice, s->stream));
    CK(cudaMemcpyAsync(s->d_prev_ub.p, s->st.ub, sizeof(double) * count, cudaMemcpyDeviceToDevice, s->stream));
    CK(cudaMemcpyAsync(s->d_prev_uid.p, s->st.inc_uid, sizeof(unsigned long long) * count, cudaMemcpyDeviceToDevice, s->stream));
    struct Shape { int C, N, R, O, E, L; };
    std::vector<Shape> prev(count);
    for (int k = 0; k < count; ++k) { const DevProb &p = s->pk.probs[k]; prev[k] = Shape{p.C, p.N, p.R, p.O, p.E, p.L}; }
    CK(cudaStreamSynchronize(s->stream));
    s->uploaded = false; s->ran = false;
    const auto tp0 = std::chrono::steady_clock::now();
    pack_batch(s, problems, count);
    const auto tp1 = std::chrono::steady_clock::now();
    upload_packed(s);
    setup_bnb(s);
    s->h_haswarm.assign(count, 0);
    for (int k = 0; k < count; ++k) {
      const DevProb &p = s->pk.probs[k];
      s->h_haswarm[k] = (p.C == prev[k].C && p.N == prev[k].N && p.R == prev[k].R && p.O == prev[k].O && p.E == prev[k].E && p.L == prev[k].L) ? 1 : 0;
    }
    CK(cudaMemcpyAsync(s->d_same.p, s->h_haswarm.data(), sizeof(int) * count, cudaMemcpyHostToDevice, s->stream));
    s->d_warm.ensure((size_t)count * s->st.ndec_stride); s->d_haswarm.ensure(count);
    launch_bnb_shift_warm(s->d_probs.p, s->d_iblob.p, count, s->d_prev_dec.p, prev_stride, s->d_prev_ub.p, s->d_prev_uid.p, s->d_same.p,
                          s->d_warm.p, s->st.ndec_stride, s->d_haswarm.p, s->stream);
    CK(cudaGetLastError());
    s->any_warm = true;
    s->stats.h2d_bytes += (long)(sizeof(int) * count);
    CK(cudaStreamSynchronize(s->stream));
    s->stats.pack_ms = std::chrono::duration<double, std::milli>(tp1 - tp0).count();
    s->stats.upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tp1).count();
    s->uploaded = true;
  } catch (const std::invalid_argument &ex) {
    return fail(s, MIQP_B200_ERR_ARG, ex.what());
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

// One search of the uploaded batch; a streaming run (s->on_done set) also harvests every plan in the round select marks it
// finished and hands it to the callback.  Both compute the same results.
static int run_batch(MiqpB200Solver *s, float *device_ms) {
  struct Reset {   // the delivered flags are seen by the kernels of streaming runs only
    MiqpB200Solver *s;
    ~Reset() { s->st.delivered = nullptr; s->on_done = nullptr; s->on_done_user = nullptr; s->hv_pending = 0; s->hv_held.clear(); }
  } reset{s};
  try {
    CK(cudaSetDevice(s->opt.device));
    start_run(s);
    run_rounds(s, -1);
    finish_run(s, device_ms);
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

int miqp_b200_batch_run(MiqpB200Solver *s, float *device_ms) {
  if (!s) return MIQP_B200_ERR_ARG;
  if (!s->uploaded) return fail(s, MIQP_B200_ERR_ARG, "batch_run without batch_upload");
  return run_batch(s, device_ms);
}

int miqp_b200_batch_run_streaming(MiqpB200Solver *s, MiqpB200PlanDone on_done, void *user, float *device_ms) {
  if (!s) return MIQP_B200_ERR_ARG;
  if (!on_done) return fail(s, MIQP_B200_ERR_ARG, "batch_run_streaming without a callback");
  if (!s->uploaded) return fail(s, MIQP_B200_ERR_ARG, "batch_run_streaming without batch_upload");
  s->on_done = on_done; s->on_done_user = user;
  return run_batch(s, device_ms);
}

static int fetch_results(MiqpB200Solver *s, double *const *x_out, double *const *traj_out, MiqpB200SolveInfo *infos);
int miqp_b200_batch_fetch(MiqpB200Solver *s, double *const *x_out, MiqpB200SolveInfo *infos) { return fetch_results(s, x_out, nullptr, infos); }
int miqp_b200_batch_fetch_compact(MiqpB200Solver *s, double *const *traj_out, MiqpB200SolveInfo *infos) { return fetch_results(s, nullptr, traj_out, infos); }

int miqp_b200_fetch_vector(MiqpB200Solver *s, int k, double *x_out) {
  if (!s || !x_out) return MIQP_B200_ERR_ARG;
  if (!s->ran || k < 0 || k >= s->st.count) return fail(s, MIQP_B200_ERR_ARG, "fetch_vector: no results for this plan index");
  const DevProb &p = s->pk.probs[k];
  if (cudaSetDevice(s->opt.device) != cudaSuccess ||
      cudaMemcpyAsync(x_out, s->d_x.p + p.x_base, sizeof(double) * p.ncols, cudaMemcpyDeviceToHost, s->stream) != cudaSuccess ||
      cudaStreamSynchronize(s->stream) != cudaSuccess) return fail(s, MIQP_B200_ERR_CUDA, "copy of the solution vector failed");
  return MIQP_B200_OK;
}

// x_out: full OPL column vectors; traj_out (compact results): [C][N][8] per plan, the incumbent trajectories as bnb_finish_kernel
// left them in inc_z.  Either may be null.
static int fetch_results(MiqpB200Solver *s, double *const *x_out, double *const *traj_out, MiqpB200SolveInfo *infos) {
  if (!s) return MIQP_B200_ERR_ARG;
  if (!s->ran) return fail(s, MIQP_B200_ERR_ARG, "batch_fetch without batch_run");
  try {
    CK(cudaSetDevice(s->opt.device));
    const int count = s->st.count;
    const long ncols = x_out ? s->pk.total_cols : 0;
    const auto tf0 = std::chrono::steady_clock::now();
    if (traj_out) {
      s->h_z.resize((size_t)count * s->st.zstride);
      CK(cudaMemcpyAsync(s->h_z.data(), s->st.inc_z, sizeof(double) * s->h_z.size(), cudaMemcpyDeviceToHost, s->stream));
    }
    s->h_x.resize(ncols); s->h_viol.resize(count); s->h_obj.resize(count); s->h_bb.resize(count); s->h_ub.resize(count);
    s->h_stats.resize((size_t)4 * count); s->h_done.resize(count); s->h_overflow.resize(count); s->h_incuid.resize(count);
    CK(cudaMemcpyAsync(s->h_incuid.data(), s->st.inc_uid, sizeof(unsigned long long) * count, cudaMemcpyDeviceToHost, s->stream));
    if (ncols > 0) CK(cudaMemcpyAsync(s->h_x.data(), s->d_x.p, sizeof(double) * ncols, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(s->h_viol.data(), s->d_viol.p, sizeof(double) * count, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(s->h_obj.data(), s->d_obj.p, sizeof(double) * count, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(s->h_bb.data(), s->d_bb.p, sizeof(double) * count, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(s->h_ub.data(), s->st.ub, sizeof(double) * count, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(s->h_stats.data(), s->b_stats.p, sizeof(unsigned long long) * 4 * count, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(s->h_done.data(), s->st.done, sizeof(int) * count, cudaMemcpyDeviceToHost, s->stream));
    s->h_doneround.resize(count);
    CK(cudaMemcpyAsync(s->h_doneround.data(), s->st.done_round, sizeof(int) * count, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(s->h_overflow.data(), s->st.overflow, sizeof(int) * count, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    s->stats.d2h_bytes = (long)(sizeof(double) * (ncols + 4 * count + (traj_out ? s->h_z.size() : 0)) + sizeof(unsigned long long) * 5 * count + 2 * sizeof(int) * count);
    if (traj_out)
      for (int k = 0; k < count; ++k) {
        const DevProb &p = s->pk.probs[k];
        if (traj_out[k]) std::memcpy(traj_out[k], s->h_z.data() + (size_t)k * s->st.zstride, sizeof(double) * (size_t)p.C * p.N * 8);
      }
    long nodes = 0, iters = 0, rows = 0;
    if (x_out) {   // scatter of the solution vectors into the caller's buffers: a few host threads for large batches
      const int nthr = (ncols * (long)sizeof(double) > (8L << 20)) ? 4 : 1;
      auto scatter = [&](int k0, int k1) {
        for (int k = k0; k < k1; ++k) {
          const DevProb &p = s->pk.probs[k];
          if (x_out[k]) std::memcpy(x_out[k], s->h_x.data() + p.x_base, sizeof(double) * p.ncols);
        }
      };
      if (nthr == 1) scatter(0, count);
      else {
        std::vector<std::thread> th;
        for (int t = 0; t < nthr; ++t) th.emplace_back(scatter, (int)((long)count * t / nthr), (int)((long)count * (t + 1) / nthr));
        for (std::thread &t : th) t.join();
      }
    }
    for (int k = 0; k < count; ++k) {
      nodes += (long)s->h_stats[k]; iters += (long)s->h_stats[count + k]; rows += (long)s->h_stats[2 * count + k];
      if (!infos) continue;
      plan_info(s, k, s->h_ub[k], s->h_incuid[k], s->h_bb[k], s->h_obj[k], s->h_viol[k], s->h_done[k], s->h_doneround[k], s->h_overflow[k],
                s->h_stats[k], s->h_stats[count + k], s->h_stats[3 * (size_t)count + k], infos[k]);
    }
    s->stats.nodes = nodes; s->stats.qp_iters = iters; s->stats.rows_visited = rows;
    s->stats.fetch_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tf0).count();
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

int miqp_b200_solve_batch_compact(MiqpB200Solver *s, const MiqpB200Problem *problems, int count, const double *const *warm,
                                  double *const *traj_out, MiqpB200SolveInfo *infos) {
  int rc = miqp_b200_batch_upload(s, problems, count, warm);
  if (rc != MIQP_B200_OK) return rc;
  rc = miqp_b200_batch_run(s, nullptr);
  if (rc != MIQP_B200_OK) return rc;
  return miqp_b200_batch_fetch_compact(s, traj_out, infos);
}

int miqp_b200_solve_batch(MiqpB200Solver *s, const MiqpB200Problem *problems, int count, const double *const *warm,
                          double *const *x_out, MiqpB200SolveInfo *infos) {
  int rc = miqp_b200_batch_upload(s, problems, count, warm);
  if (rc != MIQP_B200_OK) return rc;
  rc = miqp_b200_batch_run(s, nullptr);
  if (rc != MIQP_B200_OK) return rc;
  return miqp_b200_batch_fetch(s, x_out, infos);
}

// ---- frontier sharding: the round loop in steps, driven by the caller (one process per GPU, NCCL between them) -----------------
int miqp_b200_frontier_start(MiqpB200Solver *s) {
  if (!s) return MIQP_B200_ERR_ARG;
  if (!s->uploaded) return fail(s, MIQP_B200_ERR_ARG, "frontier_start without batch_upload");
  try {
    CK(cudaSetDevice(s->opt.device));
    start_run(s);
    CK(cudaStreamSynchronize(s->stream));
  } catch (const std::exception &ex) { return fail(s, MIQP_B200_ERR_CUDA, ex.what()); }
  return MIQP_B200_OK;
}

int miqp_b200_frontier_rounds(MiqpB200Solver *s, int nrounds, int *unfinished) {
  if (!s || !s->uploaded) return MIQP_B200_ERR_ARG;
  try {
    CK(cudaSetDevice(s->opt.device));
    const int left = run_rounds(s, nrounds);
    if (unfinished) *unfinished = s->timed_out ? 0 : left;
  } catch (const std::exception &ex) { return fail(s, MIQP_B200_ERR_CUDA, ex.what()); }
  return MIQP_B200_OK;
}

int miqp_b200_frontier_split(MiqpB200Solver *s, int rank, int world) {
  if (!s || !s->uploaded || world < 1 || rank < 0 || rank >= world) return MIQP_B200_ERR_ARG;
  try {
    CK(cudaSetDevice(s->opt.device));
    launch_bnb_split(s->st, rank, world, s->stream);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s->stream));
    ++s->fr_launches;
  } catch (const std::exception &ex) { return fail(s, MIQP_B200_ERR_CUDA, ex.what()); }
  return MIQP_B200_OK;
}

int miqp_b200_frontier_fingerprint(MiqpB200Solver *s, long long *fp) {
  if (!s || !s->uploaded || !fp) return MIQP_B200_ERR_ARG;
  try {
    CK(cudaSetDevice(s->opt.device));
    s->d_fp.ensure(s->st.count);
    launch_bnb_fingerprint(s->st, s->d_fp.p, s->stream);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(fp, s->d_fp.p, sizeof(long long) * s->st.count, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    ++s->fr_launches;
  } catch (const std::exception &ex) { return fail(s, MIQP_B200_ERR_CUDA, ex.what()); }
  return MIQP_B200_OK;
}

int miqp_b200_frontier_ub_device(MiqpB200Solver *s, void **ub, int *count) {
  if (!s || !s->uploaded || !ub) return MIQP_B200_ERR_ARG;
  *ub = s->st.ub;
  if (count) *count = s->st.count;
  return MIQP_B200_OK;
}

int miqp_b200_frontier_get_ub(MiqpB200Solver *s, double *ub) {
  if (!s || !s->uploaded || !ub) return MIQP_B200_ERR_ARG;
  if (cudaMemcpy(ub, s->st.ub, sizeof(double) * s->st.count, cudaMemcpyDeviceToHost) != cudaSuccess) return fail(s, MIQP_B200_ERR_CUDA, "copy of the incumbent objectives failed");
  return MIQP_B200_OK;
}

int miqp_b200_frontier_tighten(MiqpB200Solver *s, const double *ub) {
  if (!s || !s->uploaded || !ub) return MIQP_B200_ERR_ARG;
  try {
    CK(cudaSetDevice(s->opt.device));
    s->d_ubx.ensure(s->st.count);
    CK(cudaMemcpyAsync(s->d_ubx.p, ub, sizeof(double) * s->st.count, cudaMemcpyHostToDevice, s->stream));
    launch_bnb_tighten(s->st, s->d_ubx.p, s->stream);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s->stream));
    ++s->fr_launches;
  } catch (const std::exception &ex) { return fail(s, MIQP_B200_ERR_CUDA, ex.what()); }
  return MIQP_B200_OK;
}

int miqp_b200_frontier_finish(MiqpB200Solver *s, float *device_ms) {
  if (!s || !s->uploaded) return MIQP_B200_ERR_ARG;
  try {
    CK(cudaSetDevice(s->opt.device));
    finish_run(s, device_ms);
  } catch (const std::exception &ex) { return fail(s, MIQP_B200_ERR_CUDA, ex.what()); }
  return MIQP_B200_OK;
}

int miqp_b200_mark(MiqpB200Solver *s, int which) {
  if (!s || which < 0 || which > 1) return MIQP_B200_ERR_ARG;
  if (cudaSetDevice(s->opt.device) != cudaSuccess || cudaEventRecord(s->mark[which], s->stream) != cudaSuccess) return fail(s, MIQP_B200_ERR_CUDA, "cudaEventRecord failed");
  return MIQP_B200_OK;
}

int miqp_b200_elapsed(MiqpB200Solver *from, MiqpB200Solver *to, float *ms) {
  if (!from || !to || !ms) return MIQP_B200_ERR_ARG;
  if (cudaEventSynchronize(from->mark[0]) != cudaSuccess || cudaEventSynchronize(to->mark[1]) != cudaSuccess ||
      cudaEventElapsedTime(ms, from->mark[0], to->mark[1]) != cudaSuccess) return fail(to, MIQP_B200_ERR_CUDA, "cudaEventElapsedTime failed");
  return MIQP_B200_OK;
}

int miqp_b200_measure_fp64_peak(MiqpB200Solver *s, double *tflops) {
  if (!s || !tflops) return MIQP_B200_ERR_ARG;
  if (cudaSetDevice(s->opt.device) != cudaSuccess) return fail(s, MIQP_B200_ERR_CUDA, "cudaSetDevice failed");
  const double tf = miqp::measure_fp64_tflops(s->num_sms, s->stream, 5);
  if (tf <= 0.0) return fail(s, MIQP_B200_ERR_CUDA, "fp64 micro-benchmark failed");
  *tflops = tf;
  return MIQP_B200_OK;
}

int miqp_b200_debug_traces(MiqpB200Solver *s, double *out4096) {
  if (!s || !out4096 || !s->b_dbg.p) return MIQP_B200_ERR_ARG;
  if (cudaMemcpy(out4096, s->b_dbg.p + (size_t)1024 * 512, 8 * 512 * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess)
    return fail(s, MIQP_B200_ERR_CUDA, "trace copy failed");
  return MIQP_B200_OK;
}

int miqp_b200_debug_profile(MiqpB200Solver *s, unsigned long long *out256) {
  if (!s || !out256 || !s->b_prof.p) return MIQP_B200_ERR_ARG;
  if (cudaMemcpy(out256, s->b_prof.p, 256 * sizeof(unsigned long long), cudaMemcpyDeviceToHost) != cudaSuccess)
    return fail(s, MIQP_B200_ERR_CUDA, "profile copy failed");
  return MIQP_B200_OK;
}

// ---- solution pool --------------------------------------------------------------------------------------------------------
int miqp_b200_set_solution_pool(MiqpB200Solver *s, int capacity) {
  if (!s) return MIQP_B200_ERR_ARG;
  if (capacity < 0 || capacity > 64) return fail(s, MIQP_B200_ERR_ARG, "solution pool capacity must lie in 0..64");
  s->solution_pool = capacity;
  return MIQP_B200_OK;
}

static const char *pool_unavailable(const MiqpB200Solver *s) {
  if (!s->uploaded || !s->ran) return "solution pool: no results of a batch_run on this solver";
  if (s->st.pool_cap <= 0) return "solution pool: the pool was off when this batch was uploaded (miqp_b200_set_solution_pool)";
  return nullptr;
}

int miqp_b200_pool_sizes(MiqpB200Solver *s, int *sizes) {
  if (!s || !sizes) return MIQP_B200_ERR_ARG;
  if (const char *why = pool_unavailable(s)) return fail(s, MIQP_B200_ERR_ARG, why);
  if (cudaSetDevice(s->opt.device) != cudaSuccess ||
      cudaMemcpyAsync(sizes, s->st.pool_cnt, sizeof(int) * s->st.count, cudaMemcpyDeviceToHost, s->stream) != cudaSuccess ||
      cudaStreamSynchronize(s->stream) != cudaSuccess) return fail(s, MIQP_B200_ERR_CUDA, "copy of the solution pool sizes failed");
  return MIQP_B200_OK;
}

// Entries of plan k best first: the records are sorted by (search value, uid) on the host, the chosen entries are expanded into
// full column vectors on the device (pool_expand_kernel) and evaluated against the big-M model by evaluate_kernel.
int miqp_b200_pool_fetch(MiqpB200Solver *s, int k, int max_entries, MiqpB200PoolEntry *entries, double *x_out, double *traj_out,
                         int *n_out) {
  if (!s || !entries || !n_out || max_entries < 0) return MIQP_B200_ERR_ARG;
  if (const char *why = pool_unavailable(s)) return fail(s, MIQP_B200_ERR_ARG, why);
  if (k < 0 || k >= s->st.count) return fail(s, MIQP_B200_ERR_ARG, "pool_fetch: plan index out of range");
  try {
    CK(cudaSetDevice(s->opt.device));
    const BnbState &st = s->st;
    int cnt = 0;
    std::vector<PoolRec> rec((size_t)st.pool_cap);
    CK(cudaMemcpyAsync(&cnt, st.pool_cnt + k, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(rec.data(), st.pool_rec + (size_t)k * st.pool_cap, sizeof(PoolRec) * st.pool_cap, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    std::vector<int> idx(cnt);
    for (int e = 0; e < cnt; ++e) idx[e] = e;
    std::sort(idx.begin(), idx.end(), [&](int a, int b) {
      return rec[a].val < rec[b].val || (rec[a].val == rec[b].val && rec[a].uid < rec[b].uid);
    });
    const int n = std::min(cnt, max_entries);
    idx.resize(n);
    *n_out = n;
    if (n == 0) return MIQP_B200_OK;
    DevProb p;   // the device copy: prepare_tables_kernel completes the plan's record there
    CK(cudaMemcpyAsync(&p, s->d_probs.p + k, sizeof(DevProb), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    std::vector<DevProb> ep(n, p);
    for (int e = 0; e < n; ++e) ep[e].x_base = (long)e * p.ncols;
    s->sp_probs.ensure(n); s->sp_idx.ensure(n); s->sp_obj.ensure(n); s->sp_viol.ensure(n);
    s->sp_x.ensure((size_t)n * p.ncols); s->sp_zs.ensure((size_t)n * st.zstride);
    CK(cudaMemcpyAsync(s->sp_probs.p, ep.data(), sizeof(DevProb) * n, cudaMemcpyHostToDevice, s->stream));
    CK(cudaMemcpyAsync(s->sp_idx.p, idx.data(), sizeof(int) * n, cudaMemcpyHostToDevice, s->stream));
    launch_pool_expand(st, k, s->sp_idx.p, n, s->sp_probs.p, s->d_dblob.p, s->d_iblob.p, s->sp_zs.p, s->sp_x.p, s->stream);
    CK(cudaMemsetAsync(s->sp_viol.p, 0, sizeof(double) * n, s->stream));
    launch_evaluate(s->sp_probs.p, s->d_dblob.p, s->d_iblob.p, n, s->pk.max_rows, s->sp_x.p, s->sp_viol.p, s->sp_obj.p, s->stream);
    CK(cudaGetLastError());
    std::vector<double> obj(n), viol(n);
    CK(cudaMemcpyAsync(obj.data(), s->sp_obj.p, sizeof(double) * n, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(viol.data(), s->sp_viol.p, sizeof(double) * n, cudaMemcpyDeviceToHost, s->stream));
    if (x_out) CK(cudaMemcpyAsync(x_out, s->sp_x.p, sizeof(double) * n * p.ncols, cudaMemcpyDeviceToHost, s->stream));
    const long tsz = (long)p.C * p.N * 8;   // the trajectory part of an entry's zstride doubles
    if (traj_out)
      for (int e = 0; e < n; ++e)
        CK(cudaMemcpyAsync(traj_out + e * tsz, s->sp_zs.p + (size_t)e * st.zstride, sizeof(double) * tsz, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    for (int e = 0; e < n; ++e) {
      const PoolRec &r = rec[idx[e]];
      MiqpB200PoolEntry &o = entries[e];
      o.objective = obj[e]; o.max_violation = viol[e]; o.search_value = r.val;
      o.converged = r.converged; o.round = r.round; o.uid = r.uid;
    }
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

// ---- pool export / merge (frontier sharding: the pools of all ranks) ----------------------------------------------------------
int miqp_b200_pool_export(MiqpB200Solver *s, void **dev, size_t *bytes) {
  if (!s || !dev || !bytes) return MIQP_B200_ERR_ARG;
  if (const char *why = pool_unavailable(s)) return fail(s, MIQP_B200_ERR_ARG, why);
  try {
    CK(cudaSetDevice(s->opt.device));
    const BnbState &st = s->st;
    const PoolExportLayout l = export_layout(st);
    const PoolExportHeader h = export_header(s);
    const size_t entries = (size_t)st.count * st.pool_cap;
    s->sp_export.ensure((size_t)l.bytes);
    unsigned char *b = s->sp_export.p;
    CK(cudaMemcpyAsync(b, &h, sizeof h, cudaMemcpyHostToDevice, s->stream));
    CK(cudaMemcpyAsync(b + l.off_cnt, st.pool_cnt, sizeof(int) * st.count, cudaMemcpyDeviceToDevice, s->stream));
    CK(cudaMemcpyAsync(b + l.off_rec, st.pool_rec, sizeof(PoolRec) * entries, cudaMemcpyDeviceToDevice, s->stream));
    CK(cudaMemcpyAsync(b + l.off_dec, st.pool_dec, entries * st.ndec_stride, cudaMemcpyDeviceToDevice, s->stream));
    CK(cudaMemcpyAsync(b + l.off_z, st.pool_z, sizeof(double) * entries * st.zstride, cudaMemcpyDeviceToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));   // (the header's host copy goes out of scope)
    *dev = b;
    *bytes = (size_t)l.bytes;
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

int miqp_b200_pool_merge(MiqpB200Solver *s, const void *gathered, int world) {
  if (!s) return MIQP_B200_ERR_ARG;
  if (const char *why = pool_unavailable(s)) return fail(s, MIQP_B200_ERR_ARG, why);
  if (!gathered || world < 1) return fail(s, MIQP_B200_ERR_ARG, "pool_merge: no input or world < 1");
  if ((long)world * s->st.pool_cap > POOL_MERGE_MAX)
    return fail(s, MIQP_B200_ERR_ARG, "pool_merge: world x pool capacity exceeds " + std::to_string(POOL_MERGE_MAX));
  try {
    CK(cudaSetDevice(s->opt.device));
    const PoolExportLayout l = export_layout(s->st);
    const size_t total = (size_t)l.bytes * world;
    cudaPointerAttributes attr;
    const bool here = cudaPointerGetAttributes(&attr, gathered) == cudaSuccess && attr.device == s->opt.device &&
                      (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged);
    cudaGetLastError();   // (an older runtime reports a host pointer it does not know as an error)
    // headers first, every one checked before the pool changes
    const PoolExportHeader mine = export_header(s);
    std::vector<PoolExportHeader> hs(world);
    for (int r = 0; r < world; ++r) {
      const unsigned char *src = static_cast<const unsigned char *>(gathered) + (size_t)r * l.bytes;
      CK(cudaMemcpyAsync(&hs[r], src, sizeof(PoolExportHeader), cudaMemcpyDefault, s->stream));
    }
    CK(cudaStreamSynchronize(s->stream));
    for (int r = 0; r < world; ++r) {
      const PoolExportHeader &h = hs[r];
      if (h.magic != mine.magic || h.version != mine.version || h.count != mine.count || h.cap != mine.cap ||
          h.zstride != mine.zstride || h.ndec_stride != mine.ndec_stride || h.shape_hash != mine.shape_hash)
        return fail(s, MIQP_B200_ERR_ARG, "pool_merge: export " + std::to_string(r) +
                                              " does not come from a solver with this batch's shapes and pool capacity");
    }
    const unsigned char *g = static_cast<const unsigned char *>(gathered);
    if (!here) {   // host memory or another GPU: a copy on this solver's device
      s->sp_gathered.ensure(total);
      CK(cudaMemcpyAsync(s->sp_gathered.p, gathered, total, cudaMemcpyDefault, s->stream));
      g = s->sp_gathered.p;
    }
    launch_pool_merge(s->st, s->d_probs.p, g, l, world, s->stream);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s->stream));
    s->stats.launches += 1;
  } catch (const std::exception &ex) {
    return fail(s, MIQP_B200_ERR_CUDA, ex.what());
  }
  return MIQP_B200_OK;
}

int miqp_b200_run_stats(const MiqpB200Solver *s, MiqpB200RunStats *out) {
  if (!s || !out) return MIQP_B200_ERR_ARG;
  *out = s->stats;
  return MIQP_B200_OK;
}

}  // extern "C"
