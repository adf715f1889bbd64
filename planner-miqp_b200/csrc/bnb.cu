// bnb.cu -- device-resident branch and bound over a batch of plans.
//
// What the reference delegates to cplex.solve() (src/cplex_wrapper.cpp:158-185): a search over
// the binaries of cplexmodel/*.mod that stops at the CPLEX relative gap
// |best_bound - incumbent| / (1e-10 + |incumbent|) <= epgap (cplexmodel.mod:8-10).
//
// Every plan owns a pool of open nodes in HBM (structure of arrays, fixed capacity, free-slot
// stack).  One round of the search is two kernels:
//
//   bnb_select_kernel  one CTA per plan: releases the slots handed out in the last round,
//                      snapshots the cutoff from the incumbent, prunes the open list by
//                      bound, picks the K best nodes (radix select on 64-bit priority keys:
//                      depth first until an incumbent exists, best bound first afterwards)
//                      and appends them to the global work list.
//   bnb_nodes_kernel   persistent teams (one CTA of four warps, eight when a round holds fewer nodes than SMs) pull
//                      (plan, node) items from the work list; a team solves its node relaxation (node_qp.cuh)
//                      -- started from the parent's relaxed optimum, parked in HBM and continued next round if it
//                      needs more than its iteration budget --, warp 0 then scans the relaxed optimum for violated
//                      disjunctions and either records an incumbent or pushes the children (one per alternative
//                      of the most violated disjunction, with their lower bounds) onto the plan's pool.
//
// The host only launches rounds and polls one integer (number of unfinished plans).
#include "kernels.cuh"
#include "node_qp.cuh"
#include "bnb_common.cuh"

namespace miqp {

// priority key, smaller = earlier.  Without incumbent the search dives: the children created in the
// last round come first (least violated alternative first, then bound); if the dive died (no
// newborn node) it restarts from the best bound.  Deepest-first backtracking is deliberately NOT
// used: it gets trapped below a wrong early decision (seen on 3 of 512 config-2 plans: 20k+ nodes
// instead of ~40).  With an incumbent: best bound first, then deepest.
__device__ __forceinline__ unsigned long long node_key(double bound, int depth, int rank, unsigned long long uid, bool have_inc, bool newborn) {
  unsigned long long d = 1023 - (unsigned long long)(depth > 1023 ? 1023 : depth);  // 10 bits
  unsigned long long r = (unsigned long long)(rank + 1 > 127 ? 127 : rank + 1);      // 7 bits
  unsigned long long b = ordered_bits(bound) >> 24;                                   // 40 bits
  unsigned long long u = uid & 127ULL;                                                // 7 bits
  if (have_inc) return (b << 24) | (d << 14) | (r << 7) | u;
  if (newborn) return (r << 47) | (b << 7) | u;
  return (1ULL << 63) | (b << 17) | (d << 7) | u;
}

// ---------------------------------------------------------------------------------------
// init
// ---------------------------------------------------------------------------------------
__global__ void bnb_init_kernel(BnbState st, const DevProb *probs, const unsigned char *warm_dec, const int *has_warm) {
  const int s = blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x;
  const long pb = (long)s * st.cap;
  const int nroot = (has_warm && has_warm[s]) ? 2 : 1;
  // free stack: slots cap-1 .. nroot (top of stack = lowest index first out)
  for (int k = tid; k < st.cap - nroot; k += nt) st.free_stack[pb + k] = st.cap - 1 - k;
  unsigned char *d0 = st.dec + (pb + 0) * st.ndec_stride;
  for (int k = tid; k < st.ndec_stride; k += nt) d0[k] = UNDEC;
  if (nroot == 2) {
    unsigned char *d1 = st.dec + (pb + 1) * st.ndec_stride;
    const unsigned char *wd = warm_dec + (long)s * st.ndec_stride;
    for (int k = tid; k < st.ndec_stride; k += nt) d1[k] = wd[k];
  }
  if (tid == 0) {
    st.free_cnt[s] = st.cap - nroot;
    st.bound[pb] = -MQ_INF; st.meta[pb] = make_int2(0, meta_word(0, 0)); st.uid[pb] = 1ULL;
    st.open_idx[pb] = 0;
    if (nroot == 2) {  // MIP start: the fully decided node is evaluated first (cplex_wrapper.cpp:494-639)
      st.bound[pb + 1] = -MQ_INF; st.meta[pb + 1] = make_int2(DEPTH_MIP_START, meta_word(0, -1)); st.uid[pb + 1] = 2ULL;   // rank -1: before the root
      st.open_idx[pb + 1] = 1;
    }
    if (st.zpool) for (int r = 0; r < nroot; ++r) st.zpool[(pb + r) * (long)st.zp_stride] = __longlong_as_double(0x7ff8000000000000LL);   // no parent: cold start
    st.open_cnt[s] = nroot;
    st.sel_cnt[s] = 0;
    st.ub[s] = MQ_INF; st.cutoff[s] = MQ_INF; st.pruned_lb[s] = MQ_INF;
    st.done[s] = 0; st.done_round[s] = -1; st.lock[s] = 0;
    st.stat_nodes[s] = 0; st.stat_iters[s] = 0; st.stat_rows[s] = 0; st.stat_uncert[s] = 0; st.overflow[s] = 0;
    st.inc_uid[s] = ~0ULL;
    if (st.pool_cap > 0) st.pool_cnt[s] = 0;
    if (s == 0) { *st.active_prev = 0; *st.work_cnt = 0; *st.work_next = 0; *st.active = 0; *st.err = 0; *st.work_cnt2 = 0; *st.work_next2 = 0; }
  }
}

void launch_bnb_init(const BnbState &st, const DevProb *probs, const unsigned char *warm_dec, const int *has_warm, cudaStream_t s) {
  bnb_init_kernel<<<st.count, 128, 0, s>>>(st, probs, warm_dec, has_warm);
}

// ---------------------------------------------------------------------------------------
// select
// ---------------------------------------------------------------------------------------
constexpr int SEL_THREADS = 256;

__device__ __forceinline__ int block_excl_scan(int flag, int *warp_tot /*[8]*/, int &total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned bal = __ballot_sync(FULL, flag);
  int pre = __popc(bal & ((1u << lane) - 1));
  if (lane == 0) warp_tot[wid] = __popc(bal);
  __syncthreads();
  int off = 0; total = 0;
  for (int k = 0; k < SEL_THREADS / 32; ++k) { int t = warp_tot[k]; if (k < wid) off += t; total += t; }
  __syncthreads();
  return off + pre;
}

__global__ void __launch_bounds__(SEL_THREADS) bnb_select_kernel(BnbState st, const DevProb *probs, int round, double elapsed_s) {
  const int s = blockIdx.x;
  const int tid = threadIdx.x;
  __shared__ int warp_tot[SEL_THREADS / 32];
  __shared__ int s_out, s_free, s_tie, s_wbase, s_nsusp;
  __shared__ int hist[256];
  __shared__ double s_pruned[SEL_THREADS / 32];
  __shared__ unsigned long long s_prefix; __shared__ int s_remaining;
  if (st.done[s]) return;
  if (st.tlimit && elapsed_s > st.tlimit[s]) {   // this plan's own time limit (max_solution_time): it stops with what it has
    if (tid == 0) { st.done[s] = 2; st.done_round[s] = round - 1; st.sel_cnt[s] = 0; }
    return;
  }
  const DevProb &p = probs[s];
  const long pb = (long)s * st.cap;
  const int KS = st.sel_per_plan;   // stride of sel_idx = largest number of nodes a plan may take per round
  // 1. release the slots processed in the last round
  const int nsel_prev = st.sel_cnt[s];
  const int free0 = st.free_cnt[s];
  // (a parked relaxation keeps its node slot: it is back in the open list and continues this round)
  if (tid == 0) {
    int f = free0;
    for (int k = 0; k < nsel_prev; ++k) { const int sl = st.sel_idx[(long)s * KS + k]; if (!st.susp_slot || st.susp_slot[pb + sl] < 0) st.free_stack[pb + f++] = sl; }
    s_free = f; s_out = 0; s_tie = 0; s_nsusp = 0;
  }
  // 2. cutoff snapshot
  const double ub = st.ub[s];
  const bool have_inc = ub < MQ_INF;
  const double cutoff = have_inc ? ub - p.gap_tol * fabs(ub) : MQ_INF;
  // nodes taken this round: one dive head per plan until an incumbent exists; afterwards the base
  // count, raised when few plans are still active so that the resident warps stay busy
  int K = st.sel_dive;
  const int act = *st.active_prev > 0 ? *st.active_prev : st.count;
  const int fill = st.nwarps / act;
  if (have_inc) {
    K = st.sel_base;
    if (fill > K) K = fill;
    if (K > KS) K = KS;
  } else {
    if (st.dive_fill > 0) { const int kd = fill / st.dive_fill; if (kd > K) K = kd; }
    // still no incumbent long after the typical plan has finished its dive: a hard plan, widen its beam
    if (st.dive_patience > 0 && round > st.dive_patience) { const int kp = (round - st.dive_patience) * st.dive_growth; if (kp > K) K = kp; }
    if (K > KS) K = KS;
  }
  __syncthreads();
  // 3. prune by bound, compute keys, compact in place
  const int n0 = st.open_cnt[s];
  double pruned = MQ_INF;
  for (int base = 0; base < n0; base += SEL_THREADS) {
    const int idx = base + tid;
    int slot = -1, keep = 0; unsigned long long key = 0;
    if (idx < n0) {
      slot = st.open_idx[pb + idx];
      const double b = st.bound[pb + slot];
      keep = (b < cutoff);
      const bool parked = st.susp_slot && st.susp_slot[pb + slot] >= 0;
      if (parked && !keep) st.susp_slot[pb + slot] = -1;                 // pruned while parked
      if (parked && keep) { key = 0ULL; atomicAdd(&s_nsusp, 1); }        // continues first: its state is only kept for one round
      else if (keep) {
        int2 m = st.meta[pb + slot];
        key = node_key(b, m.x, meta_rank(m.y), st.uid[pb + slot], have_inc, meta_birth(m.y) == round - 1);
      }
      else { pruned = fmin(pruned, b); int pos = atomicAdd(&s_free, 1); st.free_stack[pb + pos] = slot; }
    }
    int total; const int rank = block_excl_scan(keep, warp_tot, total);
    const int out0 = s_out;
    if (keep) { st.open_idx[pb + out0 + rank] = slot; st.keybuf[pb + out0 + rank] = key; }
    __syncthreads();
    if (tid == 0) s_out = out0 + total;
    __syncthreads();
  }
  pruned = warp_min(pruned);
  if ((tid & 31) == 0) s_pruned[tid >> 5] = pruned;
  __syncthreads();
  const int n1 = s_out;
  if (tid == 0) {
    double pm = st.pruned_lb[s];
    for (int k = 0; k < SEL_THREADS / 32; ++k) pm = fmin(pm, s_pruned[k]);
    st.pruned_lb[s] = pm;
  }
  K += s_nsusp; if (K > KS) K = KS;   // parked relaxations do not take the place of new nodes
  // 4. threshold key of the K best
  unsigned long long T = ~0ULL; int remaining = n1;  // take everything
  if (n1 > K) {
    if (tid == 0) { s_prefix = 0ULL; s_remaining = K; }
    __syncthreads();
    for (int pass = 0; pass < 8; ++pass) {
      const int shift = 56 - 8 * pass;
      hist[tid] = 0;
      __syncthreads();
      const unsigned long long prefix = s_prefix;
      const unsigned long long himask = (pass == 0) ? 0ULL : (~0ULL << (shift + 8));
      for (int idx = tid; idx < n1; idx += SEL_THREADS) {
        const unsigned long long key = st.keybuf[pb + idx];
        if ((key & himask) == prefix) atomicAdd(&hist[(int)((key >> shift) & 255ULL)], 1);
      }
      __syncthreads();
      if (tid == 0) {
        int rem = s_remaining, b = 0;
        while (b < 255 && hist[b] < rem) { rem -= hist[b]; ++b; }
        s_remaining = rem;  // how many to take from bucket b at this digit
        s_prefix = prefix | ((unsigned long long)b << shift);
      }
      __syncthreads();
    }
    T = s_prefix; remaining = s_remaining;
  }
  // 5. hand the selected nodes to the work list, keep the rest
  __syncthreads();   // every thread has read n1 = s_out (no barrier in between when n1 <= K; racecheck finding)
  if (tid == 0) s_out = 0;
  __syncthreads();
  int nsel_total = 0;
  for (int base = 0; base < n1; base += SEL_THREADS) {
    const int idx = base + tid;
    int slot = -1, sel = 0, keep = 0; unsigned long long key = 0;
    if (idx < n1) {
      slot = st.open_idx[pb + idx]; key = st.keybuf[pb + idx];
      if (key < T) sel = 1;
      else if (key == T) sel = (atomicAdd(&s_tie, 1) < remaining);
      keep = !sel;
    }
    int tsel; const int rsel = block_excl_scan(sel, warp_tot, tsel);
    int tkeep; const int rkeep = block_excl_scan(keep, warp_tot, tkeep);
    const int out0 = s_out;
    if (sel) st.sel_idx[(long)s * KS + nsel_total + rsel] = slot;
    if (keep) { st.open_idx[pb + out0 + rkeep] = slot; st.keybuf[pb + out0 + rkeep] = key; }
    nsel_total += tsel;
    __syncthreads();
    if (tid == 0) s_out = out0 + tkeep;
    __syncthreads();
  }
  if (tid == 0) {
    st.open_cnt[s] = s_out;
    st.sel_cnt[s] = nsel_total;
    st.free_cnt[s] = s_free;
    st.cutoff[s] = cutoff;
    if (nsel_total == 0) { st.done[s] = 1; st.done_round[s] = round - 1; }  // frontier exhausted (everything pruned or solved) after the last round
    else { atomicAdd(st.active, 1); s_wbase = atomicAdd((p.C > 1 || st.force_multi) ? st.work_cnt2 : st.work_cnt, nsel_total); }
  }
  __syncthreads();
  if (nsel_total > 0) {
    const int wb = s_wbase;
    int2 *wl = (p.C > 1 || st.force_multi) ? st.work2 : st.work;   // plans with several cars go to the CTA-per-node kernel
    for (int k = tid; k < nsel_total; k += SEL_THREADS) wl[wb + k] = make_int2(s, st.sel_idx[(long)s * KS + k]);
  }
}

__global__ void bnb_round_reset_kernel(BnbState st) { if (st.susp_cnt) *st.susp_cnt = 0; *st.active_prev = *st.active; *st.work_cnt = 0; *st.work_next = 0; *st.active = 0; *st.work_cnt2 = 0; *st.work_next2 = 0; }

void launch_bnb_select(const BnbState &st, const DevProb *probs, int round, double elapsed_s, cudaStream_t s) {
  bnb_round_reset_kernel<<<1, 1, 0, s>>>(st);
  bnb_select_kernel<<<st.count, SEL_THREADS, 0, s>>>(st, probs, round, elapsed_s);
}

// ---------------------------------------------------------------------------------------
// scan of a relaxed optimum: implied alternatives and the most violated disjunction
// ---------------------------------------------------------------------------------------
struct Branch { int kind, i, o, pt; double viol; int ord; };  // kind: 0 none, 1 mode, 2 env, 3 obs
struct Fallback { int ord, kind, i, o, pt; };   // first undecided disjunction in scan order (branching of a stalled relaxation)
__device__ __forceinline__ void fb_offer(Fallback &f, int ord, int kind, int i, int o, int pt) {
  if (ord < f.ord) { f.ord = ord; f.kind = kind; f.i = i; f.o = o; f.pt = pt; }
}

__device__ __forceinline__ void branch_offer(Branch &b, double viol, int ord, int kind, int i, int o, int pt) {
  if (viol > b.viol || (viol == b.viol && ord < b.ord)) { b.viol = viol; b.ord = ord; b.kind = kind; b.i = i; b.o = o; b.pt = pt; }
}

// worst violation of the bounds (and for rho=0 modes the five mode rows) of alternative alt
__device__ __forceinline__ double mode_alt_violation(const WarpCtx &w, int i, int alt, int jprev, const double y[8]) {
  const DevProb &p = *w.p;
  double lo[8], hi[8];
  const int j = (alt == MODE_FROZEN) ? jprev : (alt >> 2);
  stage_bounds(w, i, j, alt == MODE_FROZEN, lo, hi);
  double v = -MQ_INF;
#pragma unroll
  for (int t = 1; t < 8; ++t) {
    if (t == Y_PY) continue;
    if (t >= 6 && i == w.N - 1) { if (lo[t] > 0.0) v = fmax(v, lo[t]); if (hi[t] < 0.0) v = fmax(v, -hi[t]); continue; }
    v = fmax(v, y[t] - hi[t]); v = fmax(v, lo[t] - y[t]);
  }
  if (alt != MODE_FROZEN) {
    double a[6], rhs;
#pragma unroll 1
    for (int k = 0; k < 5; ++k) {
      mode_row(w, alt >> 2, alt & 3, k, a, rhs);
      double gz = -rhs;
#pragma unroll
      for (int t = 0; t < 6; ++t) gz += a[t] * y[t];
      v = fmax(v, gz);
    }
  }
  return v;
}

__device__ __forceinline__ double edge_violation(const double *et, const double *ft, int pt, double sign, const double y[8]) {
  double a[6], rhs;
  edge_row(et, ft, pt, sign, a, rhs);
  double gz = -rhs;
#pragma unroll
  for (int t = 0; t < 6; ++t) gz += a[t] * y[t];
  return gz;
}

// returns number of undecided disjunctions; fills w.imp and br
__device__ __forceinline__ int scan_node(const WarpCtx &w, Branch &br, Fallback &fb) {
  const DevProb &p = *w.p;
  const int lane = w.lane, N = w.N, O = p.O, E = p.E, L = p.L;
  const double tol = 1e-6;
  const int ord_stride = 6 + 5 * O;
  int *bestalt = w.aux, *rdec = w.aux + N, *blame = w.aux + 2 * N;
  double *bestv = w.auxd;
  const int nalt = w.I[p.o_nalt];
  const int *alts = w.I + p.o_alt;
  for (int k = lane; k < p.ndec_pad; k += 32) w.imp[k] = w.dec[k];
  // phase 1: best rho=0 alternative per undecided stage (independent of the previous region)
  for (int i = lane; i < N; i += 32) {
    if (i == 0 || w.dec[p.off_mode + i] != UNDEC) continue;
    double y[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) y[t] = w.V[i * V_STRIDE + V_Z + t];
    int best = -1; double bv = MQ_INF;
    for (int a = 0; a < nalt; ++a) {
      const int alt = alts[a];
      const double v = mode_alt_violation(w, i, alt, 0, y);
      if (v < bv - 1e-12) { bv = v; best = alt; }
    }
    bestalt[i] = best; bestv[i] = bv;
  }
  __syncwarp();
  // phase 2: region chain (all lanes redundantly; the frozen alternative inherits the region)
  br.kind = 0; br.viol = tol; br.ord = 0x7fffffff; br.i = 0; br.o = 0; br.pt = 0;
  fb.ord = 0x7fffffff; fb.kind = 0; fb.i = 0; fb.o = 0; fb.pt = 0;
  int und = 0;
  {
    int jp = w.I[p.o_initreg] - 1;
    int root_undec = -1;
    for (int i = 1; i < N; ++i) {
      const unsigned char m = w.dec[p.off_mode + i];
      int j;
      if (m == UNDEC || (m == MODE_FROZEN && root_undec >= 0)) {
        double y[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) y[t] = w.V[i * V_STRIDE + V_Z + t];
        const double vfz = mode_alt_violation(w, i, MODE_FROZEN, jp, y);
        if (m == UNDEC) {
          ++und;
          fb_offer(fb, i * ord_stride, 1, i, 0, 0);
          int best = MODE_FROZEN; double bv = vfz;
          if (bestalt[i] >= 0 && bestv[i] < vfz - 1e-12) { best = bestalt[i]; bv = bestv[i]; }
          if (lane == 0) w.imp[p.off_mode + i] = (unsigned char)best;
          j = (best == MODE_FROZEN) ? jp : (best >> 2);
          root_undec = (best == MODE_FROZEN && root_undec >= 0) ? root_undec : i;
          branch_offer(br, bv, i * ord_stride, 1, i, 0, 0);
        } else {
          j = jp;  // decided frozen, but its region is only implied: blame the chain root
          branch_offer(br, vfz, i * ord_stride, 1, root_undec, 0, 0);
        }
      } else if (m == MODE_FROZEN) {
        j = jp;
      } else { j = m >> 2; root_undec = -1; }
      if (lane == 0) { w.jeff[i] = j; rdec[i] = (root_undec < 0); blame[i] = root_undec; }
      jp = j;
    }
  }
  __syncwarp();
  // phase 3: environment polygons and obstacle edges per point (lane = stage)
  Branch mine = br;  // every lane starts from the (identical) mode result
  int und3 = 0;
  for (int i = lane; i < N; i += 32) {
    if (i == 0) continue;
    double y[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) y[t] = w.V[i * V_STRIDE + V_Z + t];
    const int j = w.jeff[i];
    const bool region_decided = rdec[i] != 0;
    const int mode_blame = blame[i];
    const double *ft = w.D + p.o_fronttab + 12 * j;
    if (E > 0)
      for (int pt = 0; pt < 5; ++pt) {
        const unsigned char d = (E == 1) ? (unsigned char)0 : w.dec[p.off_env + i * 5 + pt];
        if (d == UNDEC) { ++und3; fb_offer(fb, i * ord_stride + 1 + pt, 2, i, 0, pt); }
        if (d != UNDEC && (pt == 0 || region_decided)) continue;
        int best = -1; double bv = MQ_INF;
        for (int e = 0; e < E; ++e) {
          if (d != UNDEC && e != d) continue;
          double v = -MQ_INF;
          for (int ed = w.I[p.o_env_off + e]; ed < w.I[p.o_env_off + e + 1]; ++ed)
            v = fmax(v, edge_violation(w.D + p.o_envtab + 3 * ed, ft, pt, -1.0, y));
          if (v < bv) { bv = v; best = e; }
        }
        if (E > 1) w.imp[p.off_env + i * 5 + pt] = (unsigned char)best;
        if (pt > 0 && !region_decided) branch_offer(mine, bv, i * ord_stride + 1 + pt, 1, mode_blame, 0, 0);
        else branch_offer(mine, bv, i * ord_stride + 1 + pt, 2, i, 0, pt);
      }
    for (int o = 0; o < O; ++o)
      for (int pt = 0; pt < 5; ++pt) {
        const unsigned char d = w.dec[p.off_obs + (o * N + i) * 5 + pt];
        if (d == OBS_SOFT) continue;
        if (d == UNDEC) { ++und3; fb_offer(fb, i * ord_stride + 6 + o * 5 + pt, 3, i, o, pt); }
        if (d != UNDEC && (pt == 0 || region_decided)) continue;
        const int ne = w.I[p.o_obs_nedges + o * N + i];
        int best = -1; double bv = MQ_INF;
        for (int ed = 0; ed < ne; ++ed) {
          if (d != UNDEC && ed != d) continue;
          const double v = edge_violation(w.D + p.o_obstab + 3 * ((o * N + i) * L + ed), ft, pt, 1.0, y);
          if (v < bv) { bv = v; best = ed; }
        }
        if (ne == 0) { bv = -1.0; best = 0; }
        w.imp[p.off_obs + (o * N + i) * 5 + pt] = (unsigned char)best;
        if (pt > 0 && !region_decided) branch_offer(mine, bv, i * ord_stride + 6 + o * 5 + pt, 1, mode_blame, 0, 0);
        else branch_offer(mine, bv, i * ord_stride + 6 + o * 5 + pt, 3, i, o, pt);
      }
  }
  // phase 4: most violated, first in scan order among equals
  for (int off = 16; off > 0; off >>= 1) {
    Branch o;
    o.viol = __shfl_xor_sync(FULL, mine.viol, off); o.ord = __shfl_xor_sync(FULL, mine.ord, off);
    o.kind = __shfl_xor_sync(FULL, mine.kind, off); o.i = __shfl_xor_sync(FULL, mine.i, off);
    o.o = __shfl_xor_sync(FULL, mine.o, off); o.pt = __shfl_xor_sync(FULL, mine.pt, off);
    branch_offer(mine, o.viol, o.ord, o.kind, o.i, o.o, o.pt);
  }
  br = mine;
  for (int off = 16; off > 0; off >>= 1) {
    const int oo = __shfl_xor_sync(FULL, fb.ord, off), ok = __shfl_xor_sync(FULL, fb.kind, off), oi = __shfl_xor_sync(FULL, fb.i, off);
    const int ob = __shfl_xor_sync(FULL, fb.o, off), op = __shfl_xor_sync(FULL, fb.pt, off);
    fb_offer(fb, oo, ok, oi, ob, op);
  }
  und += warp_sum_i(und3);
  __syncwarp();
  return und;
}

// ---------------------------------------------------------------------------------------
// lower bound of a child before it is solved (derivation: bnb_multi_core.cuh, tables:
// formulation_tables.cuh): the parent's optimum z* violates a row g.z <= h of the child's
// alternative by v > 0, hence every point of the child costs at least
// f(z*) + 1/2 v^2 / (g' W_i g).  Children whose bound reaches the cutoff are never created.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double quad_w(const WarpCtx &w, int i, const double a[6]) {
  const double *t = w.D + w.p->o_wtab + 14 * i;
  double g = 0.0;
#pragma unroll
  for (int ax = 0; ax < 2; ++ax) {
    const double *m = t + 7 * ax; const double *v = a + 3 * ax;
    g += m[0] * v[0] * v[0] + 2.0 * m[1] * v[1] * v[0] + m[2] * v[1] * v[1] + 2.0 * m[3] * v[2] * v[0] + 2.0 * m[4] * v[2] * v[1] + m[5] * v[2] * v[2];
  }
  return g;
}
__device__ __forceinline__ double delta_of(double viol, double G) {
  if (!(viol > 1e-7) || !(G > 1e-14)) return 0.0;
  return 0.5 * viol * viol / G;
}
__device__ __forceinline__ double bound_delta(const WarpCtx &w, int i, int T, double viol) {
  const double *t = w.D + w.p->o_wtab + 14 * i;
  double G;
  if (T < 6) { const int o = T % 3; G = t[7 * (T / 3) + (o == 0 ? 0 : o == 1 ? 2 : 5)]; }
  else G = t[7 * (T - 6) + 6];
  return delta_of(viol, G);
}
__device__ __forceinline__ double alt_delta(const WarpCtx &w, const Branch &br, int alt) {
  const DevProb &p = *w.p;
  const int N = w.N, i = br.i;
  const int *rdec = w.aux + N;
  double y[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) y[t] = w.V[i * V_STRIDE + V_Z + t];
  double dl = 0.0, a[6], rhs;
  if (br.kind == 1) {
    const bool frozen = (alt == MODE_FROZEN);
    const int j = frozen ? ((i - 1 == 0 || rdec[i - 1]) ? w.jeff[i - 1] : -1) : (alt >> 2);
    double lo[8], hi[8];
    stage_bounds(w, i, j, frozen, lo, hi);
#pragma unroll
    for (int t = 1; t < 8; ++t) {
      if (t == Y_PY) continue;
      if (t >= 6 && i == N - 1) continue;
      dl = fmax(dl, bound_delta(w, i, t, y[t] - hi[t]));
      dl = fmax(dl, bound_delta(w, i, t, lo[t] - y[t]));
    }
    if (!frozen) {
#pragma unroll 1
      for (int k = 0; k < 5; ++k) { mode_row(w, alt >> 2, alt & 3, k, a, rhs); dl = fmax(dl, delta_of(dot6(a, y) - rhs, quad_w(w, i, a))); }
    }
  } else if (br.kind == 2) {
    const double *ft = w.D + p.o_fronttab + 12 * (w.jeff[i] >= 0 ? w.jeff[i] : 0);
    for (int ed = w.I[p.o_env_off + alt]; ed < w.I[p.o_env_off + alt + 1]; ++ed) {
      edge_row(w.D + p.o_envtab + 3 * ed, ft, br.pt, -1.0, a, rhs);
      dl = fmax(dl, delta_of(dot6(a, y) - rhs, quad_w(w, i, a)));
    }
  } else if (br.kind == 3) {
    if (alt == OBS_SOFT) return p.w_slack_obs;
    const double *ft = w.D + p.o_fronttab + 12 * (w.jeff[i] >= 0 ? w.jeff[i] : 0);
    edge_row(w.D + p.o_obstab + 3 * ((br.o * N + i) * p.L + alt), ft, br.pt, 1.0, a, rhs);
    dl = delta_of(dot6(a, y) - rhs, quad_w(w, i, a));
  }
  return dl;
}

// ---------------------------------------------------------------------------------------
// node kernel
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void effective_regions(const WarpCtx &w) {
  const DevProb &p = *w.p;
  if (w.lane == 0) {
    int jp = w.I[p.o_initreg] - 1;
    w.jeff[0] = jp;
    for (int i = 1; i < w.N; ++i) {
      const unsigned char m = w.dec[p.off_mode + i];
      int j = (m == UNDEC) ? -1 : (m == MODE_FROZEN) ? jp : (m >> 2);
      w.jeff[i] = j; jp = j;
    }
  }
  __syncwarp();
}

// shared memory of one node: S[N][S_STRIDE] V[N][V_STRIDE] T[T_SIZE] auxd[N] | rows[kmax+1][NP] (16-byte
// aligned, NP = padded stage stride, node_qp.cuh:team_row_stride) | jeff[N] aux[3N] | dec imp alternatives
struct NodeSmem { int off_rows, off_int, off_dec, total; };
// np: bound of the padded stage stride of the (s, lambda) records (team_row_stride; maxN + 7 covers every team size)
__host__ __device__ inline NodeSmem node_smem_layout(int maxN, int kmax, int ndec_stride, int np) {
  NodeSmem L;
  int b = (maxN * (S_STRIDE + V_STRIDE + 1 + 12) + T_SIZE) * 8;   // S, V, auxd, bnd (12 bound rows per stage), T
  b = (b + 15) & ~15;
  L.off_rows = b;   // (s, lambda) records: see RowIO (node_qp.cuh)
  b += (kmax + 1) * np * 16;
  L.off_int = b; b += maxN * 4 * 4;
  b = (b + 15) & ~15;
  L.off_dec = b; b += 2 * ndec_stride + 272;
  L.total = (b + 15) & ~15;
  return L;
}
int node_kernel_smem_per_warp(int maxN, int kmax, int ndec_stride) { return node_smem_layout(maxN, kmax, ndec_stride, maxN + 7).total; }
int node_kernel_narrow_np(int N) { return team_row_stride(N, team_sublanes(N, NODE_TEAM_WARPS_NARROW)); }
// two-warp teams on a batch whose single-car plans all have N steps: the records use the stride of that team size only
int node_kernel_smem_narrow(int N, int kmax, int ndec_stride) { return node_smem_layout(N, kmax, ndec_stride, team_row_stride(N, team_sublanes(N, NODE_TEAM_WARPS_NARROW))).total; }

// One CTA = one team of NODE_TEAM_WARPS warps = one node relaxation at a time (persistent: teams pull
// (plan, node) items from the round's work list).  255 registers x 128 threads x 2 CTAs fill the
// register file of an SM; the third CTA that shared memory would allow (57 kB per node at N = 40) does not fit.
// NW = 8 (one CTA per SM, 6 sub-lanes per stage at N = 40) is launched for rounds that hold fewer nodes than SMs: the
// round time is then the latency of its slowest node, and the wider team shortens the row passes.
// NW = 2 (four CTAs per SM: 255 registers x 64 threads x 4; 51 kB of shared memory per node at N = 40) is the throughput variant
// for rounds with more nodes than the four-warp teams hold at once: a node takes about 1.5x longer on two warps, twice as many are
// in flight.
template <int NW>
__global__ void __launch_bounds__(NW * 32, NW == 4 ? NODE_TEAMS_PER_SM : NW == 2 ? 4 : 1) bnb_nodes_kernel(BnbState st, const DevProb *probs, const double *dblob,
                                                                                            const int *iblob, int smem_per_node, int maxN, int row_np, int round) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double s_red[32];
  __shared__ int s_wi;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  unsigned char *base = smem_raw;
  const NodeSmem L = node_smem_layout(maxN, st.kmax, st.ndec_stride, row_np);
  WarpCtx w;
  w.D = dblob; w.I = iblob; w.lane = lane; w.wid = wid; w.nw = nw; w.red = s_red;
  const WarpGroup g{lane};   // warp 0 handles the solved node
  w.dbgrow = nullptr; w.tau_k = st.tau_k;
#ifdef MQ_PROF
  if (st.dbg && blockIdx.x < 1024) w.dbgrow = st.dbg + (size_t)blockIdx.x * 512;
#endif
  w.S = reinterpret_cast<double *>(base);
  w.V = w.S + maxN * S_STRIDE;
  w.T = w.V + maxN * V_STRIDE;
  w.auxd = w.T + T_SIZE;
  w.bnd = w.auxd + maxN; w.NB = maxN;
  w.rows = reinterpret_cast<double2 *>(base + L.off_rows);
  w.jeff = reinterpret_cast<int *>(base + L.off_int);
  w.aux = w.jeff + maxN;
  w.dec = base + L.off_dec;
  w.imp = w.dec + st.ndec_stride;
  unsigned char *alts = w.imp + st.ndec_stride;
  const int nwork = *reinterpret_cast<volatile int *>(st.work_cnt);

  for (;;) {
    __syncthreads();   // warp 0 has finished the previous node (scan, children) before its shared memory is reused
    if (threadIdx.x == 0) s_wi = atomicAdd(st.work_next, 1);
    __syncthreads();
    const int wi = s_wi;
    if (wi >= nwork) break;
    const int2 item = st.work[wi];
    const int s = item.x, slot = item.y;
    const DevProb &p = probs[s];
    const long pb = (long)s * st.cap;
    w.p = &p; w.N = p.N;
    w.sg = team_sublanes(p.N, nw); w.spw = 32 / w.sg; w.ls = lane / w.sg; w.g = lane - w.ls * w.sg;
    { const int even = (p.N + nw - 1) / nw; if (even < w.spw) w.spw = even; }   // stages spread evenly over the warps (two warps, N = 40: 20 + 20, not 32 + 8)
    w.sgmul = 65536 / w.sg + 1; w.NP = team_row_stride(p.N, w.sg); w.kmax = st.kmax;
    double pen = 0.0;
    if (wid == 0) {
      copy_dec(g, w.dec, st.dec + (pb + slot) * st.ndec_stride, st.ndec_stride);
      __syncwarp();
      effective_regions(w);
      // constant cost of SOFT obstacle decisions
      int nsoft = 0;
      for (int k = lane; k < 5 * p.O * p.N; k += 32) nsoft += (w.dec[p.off_obs + k] == OBS_SOFT);
      nsoft = warp_sum_i(nsoft);
      pen = nsoft * p.w_slack_obs;
    }
    __syncthreads();
    fill_stage_bounds(w);
    __syncthreads();

    PhiEntry e1, e2;
    e1.setup(p, lane);
    e2.setup(p, lane < 4 ? 32 + lane : 35);   // second entry of lanes 0..3: 32..35 (riccati_factor)
#ifdef MQ_PROF
    const long long pt0 = clock64();
#endif
    const double *zw = st.zpool ? st.zpool + (pb + slot) * (long)st.zp_stride : nullptr;
    if (zw && !(zw[0] == zw[0])) zw = nullptr;   // NaN marks a node without parent optimum
    SuspendIO sio;
    sio.resume = nullptr; sio.pool = nullptr; sio.counter = st.susp_cnt; sio.nslots = st.susp_slots; sio.stride = st.susp_stride; sio.budget = st.susp_budget;
    if (st.susp_slot) {
      const int ss = st.susp_slot[pb + slot];
      if (ss >= 0 && ss != SUSP_REQUEUE) sio.resume = st.susp_pool[(round + 1) & 1] + (long)ss * st.susp_stride;   // parked by the previous round
      sio.pool = st.susp_pool[round & 1];
    }
    QpResult r = solve_node_qp(w, e1, e2, zw, st.warm_mu, sio);
    // A relaxation that stalls from the parent's optimum (or after it was parked) with a feasible point well above its Lagrangian
    // bound goes back to the open list and is solved from the cold start in the next round: a stalled leaf otherwise leaves a
    // slightly suboptimal incumbent behind (scenario seed 4774: 11.8390 instead of 11.8211, reported unproven), and the cold start
    // converges where the warm one does not.  The slot is protected like a parked one (mark SUSP_REQUEUE); the NaN in its copy of
    // the parent's optimum makes the next solve a cold one, which is final.
    if (st.susp_slot && zw != nullptr &&
        ((r.status == 4) || (r.status == 0 && !r.converged && !(r.obj - r.lb <= 0.25 * p.gap_tol * fabs(r.obj))))) {
      if (threadIdx.x == 0) {
        st.zpool[(pb + slot) * (long)st.zp_stride] = __longlong_as_double(0x7ff8000000000000LL);
        st.susp_slot[pb + slot] = SUSP_REQUEUE;
        const int opos = atomicAdd(&st.open_cnt[s], 1);
        st.open_idx[pb + opos] = slot;
        atomicAdd(&st.stat_iters[s], (unsigned long long)r.iters);
        atomicAdd(&st.stat_rows[s], (unsigned long long)r.rows);
      }
      continue;
    }
    if (r.status == 3) {
      // parked: the node stays open (its bound still counts) and continues in the next round
      if (threadIdx.x == 0) {
        st.susp_slot[pb + slot] = r.susp_index;
        const int opos = atomicAdd(&st.open_cnt[s], 1);
        st.open_idx[pb + opos] = slot;
        atomicAdd(&st.stat_iters[s], (unsigned long long)r.iters);
        atomicAdd(&st.stat_rows[s], (unsigned long long)r.rows);
      }
      continue;
    }
    if (threadIdx.x == 0 && st.susp_slot) st.susp_slot[pb + slot] = -1;
    if (wid != 0) continue;
    // ---- warp 0: bookkeeping, scan of the relaxed optimum, children ----
    const double nbound = st.bound[pb + slot];
    const int2 nmeta = st.meta[pb + slot];
    const unsigned long long nuid = st.uid[pb + slot];
    const double cutoff = st.cutoff[s];
#ifdef MQ_PROF
    if (lane == 0) {
      atomicAdd(&st.prof[r.iters > 100 ? 100 : r.iters], 1ULL);
      atomicAdd(&st.prof[128], (unsigned long long)r.c_rows); atomicAdd(&st.prof[129], (unsigned long long)r.c_factor);
      atomicAdd(&st.prof[130], (unsigned long long)r.c_sweeps); atomicAdd(&st.prof[131], (unsigned long long)(clock64() - pt0));
      if (r.status != 0) { atomicAdd(&st.prof[132], 1ULL); atomicAdd(&st.prof[133], (unsigned long long)r.iters); atomicAdd(&st.prof[150 + (r.iters > 100 ? 100 : r.iters)], 1ULL); }
      if (w.dbgrow && ((r.iters >= 30 && r.status == 0) || (r.status == 0 && !r.converged) || r.status == 4)) {   // keep the traces of the first eight slow / stalled relaxations
        const unsigned long long k = atomicAdd(&st.prof[140], 1ULL);
        if (k < 8) { double *dst = st.dbg + (size_t)(1024 + k) * 512; dst[0] = r.iters; dst[1] = r.obj; dst[2] = nmeta.x; for (int q = 8; q < 8 + 5 * 100; ++q) dst[q] = w.dbgrow[q]; }
      }
      atomicAdd(&st.prof[134], (unsigned long long)r.c_a); atomicAdd(&st.prof[135], (unsigned long long)r.c_ared); atomicAdd(&st.prof[136], (unsigned long long)r.c_d);
      atomicAdd(&st.prof[137], (unsigned long long)r.c_e); atomicAdd(&st.prof[138], (unsigned long long)r.c_g); atomicAdd(&st.prof[139], (unsigned long long)r.c_atr);
    }
#endif
    if (lane == 0) count_node(st, s, r.iters, r.rows);
    if (r.status == 1) continue;  // proven infeasible (empty box or Farkas certificate): the node dies
    if (r.status != 0) { if (lane == 0) close_uncertified(st, s, nbound); continue; }
    // fval: objective of the point in V_Z (an upper bound of the relaxation); obj: lower bound of the node.  They coincide
    // when the interior-point iteration converged; a stalled iteration yields the Lagrangian bound of its multipliers.
    const double fval = r.obj + pen;
    double obj = r.converged ? fval : fmax(nbound, r.lb + pen);
    if (obj < nbound) obj = nbound;  // numerical monotonicity
    if (obj >= cutoff) { if (lane == 0) atomic_min_double(&st.pruned_lb[s], obj); continue; }
#ifdef MQ_PROF
    if (lane == 0 && !r.converged) atomicAdd(&st.prof[149], 1ULL);
#endif

    Branch br; Fallback fb;
    const int und = scan_node(w, br, fb);
    if (br.kind == 0 && und > 0 && !r.converged) {
      // The stalled point satisfies an alternative of every disjunction without being the optimum of the relaxation.  The
      // node is still replaced by the completion `imp` alone (branching on the hundreds of disjunctions that a trajectory
      // satisfies anyway would never end); the other completions are dropped, so their bound obj stays in the books: the plan
      // is reported as proven only if the incumbent comes within the gap of it.
      if (lane == 0) atomic_min_double(&st.pruned_lb[s], obj);
    }
    const Traj t = {w.V + V_Z, V_STRIDE, 1, p.N, nullptr, 0, 0};
    if (br.kind == 0 && und == 0) {   // every disjunction decided and satisfied: incumbent candidate
      offer_leaf(g, st, s, w.dec, t, fval > obj ? fval : obj, obj, r.converged, true, nuid, round);
      continue;
    }
    // children
    int nalt = 1, soff = -1;
    const unsigned char *src = w.imp;
    if (br.kind != 0) { nalt = branch_alts(p, w.I, br.kind, 0, br.i, br.o, br.pt, 0, 0, soff, lane == 0 ? alts : nullptr); src = w.dec; }
    __syncwarp();
    // child bounds (lane = alternative); the (s, lambda) records are dead after the QP solve and
    // serve as scratch.  Children that reach the cutoff are dropped.
    double *cb = reinterpret_cast<double *>(w.rows);
    if (br.kind == 0) { if (lane == 0) cb[0] = obj; }
    else for (int a = lane; a < nalt; a += 32) cb[a] = r.converged ? fmax(obj, fval + 0.999 * alt_delta(w, br, alts[a])) : obj;
    __syncwarp();
    {
      int nk = 0; double pm;
      if (lane == 0) {
        nk = drop_cut_children(alts, cb, nalt, cutoff, pm);
        if (pm < MQ_INF) atomic_min_double(&st.pruned_lb[s], pm);
      }
      nalt = __shfl_sync(FULL, nk, 0);
    }
    __syncwarp();
    if (nalt == 0) continue;
    // (the children start their interior-point solves from this node's relaxed optimum)
    push_children(g, st, s, round, nmeta.x, nuid, obj, nalt, src, 0, nullptr, soff, alts, cb, w.imp, st.zpool ? &t : nullptr);
  }
}

int node_kernel_max_ctas(int smem_per_cta, int threads) {
  int nb = 0;
  const void *fn = (threads == NODE_TEAM_WARPS_WIDE * 32) ? (const void *)bnb_nodes_kernel<NODE_TEAM_WARPS_WIDE>
                 : (threads == NODE_TEAM_WARPS_NARROW * 32) ? (const void *)bnb_nodes_kernel<NODE_TEAM_WARPS_NARROW>
                 : (const void *)bnb_nodes_kernel<NODE_TEAM_WARPS>;
  if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_per_cta) != cudaSuccess) { cudaGetLastError(); return 0; }
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, threads, smem_per_cta) != cudaSuccess) { cudaGetLastError(); return 0; }
  return nb;
}

int launch_bnb_nodes(const BnbState &st, const DevProb *probs, const double *dblob, const int *iblob,
                     int smem_per_node, int warps_per_cta, int ctas, int maxN, int row_np, int round, cudaStream_t s) {
  if (warps_per_cta == NODE_TEAM_WARPS_WIDE)
    bnb_nodes_kernel<NODE_TEAM_WARPS_WIDE><<<ctas, warps_per_cta * 32, (size_t)smem_per_node, s>>>(st, probs, dblob, iblob, smem_per_node, maxN, row_np, round);
  else if (warps_per_cta == NODE_TEAM_WARPS_NARROW)
    bnb_nodes_kernel<NODE_TEAM_WARPS_NARROW><<<ctas, warps_per_cta * 32, (size_t)smem_per_node, s>>>(st, probs, dblob, iblob, smem_per_node, maxN, row_np, round);
  else
    bnb_nodes_kernel<NODE_TEAM_WARPS><<<ctas, warps_per_cta * 32, (size_t)smem_per_node, s>>>(st, probs, dblob, iblob, smem_per_node, maxN, row_np, round);
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
// frontier sharding over several GPUs (SURVEY section 8(e).2): every rank runs the same deterministic ramp-up, then keeps
// the open nodes whose uid hashes to it; only incumbent objectives travel between the ranks afterwards
// ---------------------------------------------------------------------------------------
__global__ void bnb_split_kernel(BnbState st, int rank, int world) {
  const int s = blockIdx.x;
  if (threadIdx.x != 0 || st.done[s]) return;   // (open lists are a few hundred entries after the ramp-up: one thread per plan)
  const long pb = (long)s * st.cap;
  const int n = st.open_cnt[s];
  int keep = 0, f = st.free_cnt[s];
  for (int k = 0; k < n; ++k) {
    const int slot = st.open_idx[pb + k];
    if ((int)(mix64(st.uid[pb + slot]) % (unsigned long long)world) == rank) { st.open_idx[pb + keep++] = slot; continue; }
    // another rank owns this subtree: its bound is accounted for there.  A parked relaxation is still listed in sel_idx of the
    // last round: the next select releases its slot once the parking mark is gone (no second push here).
    if (st.susp_slot && st.susp_slot[pb + slot] >= 0) st.susp_slot[pb + slot] = -1;
    else st.free_stack[pb + f++] = slot;
  }
  st.open_cnt[s] = keep; st.free_cnt[s] = f;
}
// fingerprint of every open list (count and sum of the node uids): the ranks compare them before the split -- the ramp-up has
// to be identical everywhere, otherwise a subtree could be dropped by every rank
__global__ void bnb_fingerprint_kernel(BnbState st, unsigned long long *out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= st.count) return;
  const long pb = (long)s * st.cap;
  unsigned long long h = (unsigned long long)st.open_cnt[s] * 0x9e3779b97f4a7c15ULL;
  if (!st.done[s]) for (int k = 0; k < st.open_cnt[s]; ++k) h += mix64(st.uid[pb + st.open_idx[pb + k]]);
  out[s] = h >> 1;   // (fits a signed 64-bit integer: the caller reduces it with min / max)
}
void launch_bnb_fingerprint(const BnbState &st, unsigned long long *out, cudaStream_t s) { bnb_fingerprint_kernel<<<(st.count + 127) / 128, 128, 0, s>>>(st, out); }
void launch_bnb_split(const BnbState &st, int rank, int world, cudaStream_t s) { bnb_split_kernel<<<st.count, 32, 0, s>>>(st, rank, world); }

// incumbent objectives found elsewhere tighten the cutoff of this rank (the trajectory stays with its owner)
__global__ void bnb_tighten_kernel(BnbState st, const double *ub) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < st.count && ub[s] < st.ub[s]) st.ub[s] = ub[s];
}
void launch_bnb_tighten(const BnbState &st, const double *ub, cudaStream_t s) { bnb_tighten_kernel<<<(st.count + 127) / 128, 128, 0, s>>>(st, ub); }

// ---------------------------------------------------------------------------------------
// receding-horizon warm start on the device (MiqpPlanner::CalculateWarmstart / EnvironmentWarmstart, src/miqp_planner.cpp:787-1115,
// and the MIP start of src/cplex_wrapper.cpp:494-639): the incumbent of the previous planning cycle is kept as one decision byte per
// disjunction, so "shift every family by one step, repeat the last column, re-derive the binaries" is a shift of the bytes along the
// time axis; the last step stays undecided (the repeated column is often infeasible there) and the search completes it.  A region
// that is no longer reachable in the new cycle (possible_region moves with the car's orientation) leaves its step undecided.
// One CTA per plan; prev_* are copies of the previous cycle's incumbents, taken before the new batch was set up.
// ---------------------------------------------------------------------------------------
__global__ void bnb_shift_warm_kernel(const DevProb *probs, const int *iblob, int count, const unsigned char *prev_dec, int prev_stride,
                                      const double *prev_ub, const unsigned long long *prev_uid, const int *same_shape,
                                      unsigned char *warm_dec, int stride, int *has_warm) {
  const int s = blockIdx.x;
  if (s >= count) return;
  const DevProb &p = probs[s];
  const int *I = iblob;
  const bool ok = same_shape[s] && prev_ub[s] < MQ_INF && prev_uid[s] != ~0ULL;
  unsigned char *w = warm_dec + (long)s * stride;
  for (int e = threadIdx.x; e < stride; e += blockDim.x) w[e] = UNDEC;
  if (threadIdx.x == 0) has_warm[s] = ok ? 1 : 0;
  if (!ok) return;
  __syncthreads();
  const unsigned char *d = prev_dec + (long)s * prev_stride;
  const int C = p.C, N = p.N, O = p.O, E = p.E, P = p.P, R = p.R;
  // mode of (car, step): alternative j*4+h must exist in the new cycle, else another speed half-plane of the same region, else undecided
  for (int e = threadIdx.x; e < C * (N - 1); e += blockDim.x) {
    const int c = e / (N - 1), i = e % (N - 1);          // new step i takes old step i + 1
    if (i == 0) continue;                                 // step 0 is the fixed state
    unsigned char m = d[p.off_mode + c * N + i + 1];
    if (m != UNDEC && m != MODE_FROZEN) {
      const int na = I[p.o_nalt + c]; const int *alts = I + p.o_alt + c * 4 * R;
      int exact = 0, same_region = -1;
      for (int a = 0; a < na; ++a) { if (alts[a] == m) exact = 1; else if ((alts[a] >> 2) == (m >> 2) && same_region < 0) same_region = alts[a]; }
      if (!exact) m = (same_region >= 0) ? (unsigned char)same_region : (unsigned char)UNDEC;
    }
    w[p.off_mode + c * N + i] = m;
  }
  if (E > 1)
    for (int e = threadIdx.x; e < C * (N - 1) * 5; e += blockDim.x) {
      const int pt = e % 5, ci = e / 5, c = ci / (N - 1), i = ci % (N - 1);
      const unsigned char v = d[p.off_env + (c * N + i + 1) * 5 + pt];
      w[p.off_env + (c * N + i) * 5 + pt] = (v < E) ? v : (unsigned char)UNDEC;
    }
  for (int e = threadIdx.x; e < C * O * (N - 1) * 5; e += blockDim.x) {
    const int pt = e % 5, r = e / 5, i = r % (N - 1), co = r / (N - 1);
    unsigned char v = d[p.off_obs + (co * N + i + 1) * 5 + pt];   // the obstacle prediction moves one step ahead with the horizon
    const int o = co % O;
    if (v == OBS_SOFT) { if (I[p.o_obs_soft + o] != 1) v = UNDEC; }
    else if (v != UNDEC && v >= I[p.o_obs_nedges + o * N + i]) v = UNDEC;
    w[p.off_obs + (co * N + i) * 5 + pt] = v;
  }
  for (int e = threadIdx.x; e < P * (N - 1) * 4; e += blockDim.x) {
    const int q = e % 4, r = e / 4, i = r % (N - 1), pr = r / (N - 1);
    w[p.off_pair + (pr * N + i) * 4 + q] = d[p.off_pair + (pr * N + i + 1) * 4 + q];
  }
}
void launch_bnb_shift_warm(const DevProb *probs, const int *iblob, int count, const unsigned char *prev_dec, int prev_stride, const double *prev_ub,
                           const unsigned long long *prev_uid, const int *same_shape, unsigned char *warm_dec, int stride, int *has_warm, cudaStream_t s) {
  bnb_shift_warm_kernel<<<count, 128, 0, s>>>(probs, iblob, count, prev_dec, prev_stride, prev_ub, prev_uid, same_shape, warm_dec, stride, has_warm);
}

// ---------------------------------------------------------------------------------------
// finish: best bound, full column vector of the incumbent (collectRawResults,
// src/cplex_wrapper.cpp:311-448)
// ---------------------------------------------------------------------------------------
// Full OPL column vector x (zeroed by the caller) of a fully decided node: decisions `dec`, relaxed optimum `z` ([C][N][8], then
// the pair slacks [P][N][4]; z is overwritten with the exact trajectory).  Called by every thread of the block; jeff_s: shared
// [8 * 64].  Out of line: the incumbent (bnb_finish_kernel) and the pool entries (pool_expand_kernel) run the same code.
__device__ __noinline__ void expand_solution(const DevProb &p, const double *D, const int *I, const unsigned char *dec, double *z,
                                             double *x, int *jeff_s) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const int C = p.C, N = p.N, R = p.R, E = p.E, O = p.O, L = p.L;
  // exact trajectory from the jerks (model_region_constraints.mod:11-19)
  if (tid < C) {
    const int c = tid;
    double *zc = z + (long)c * N * 8;
    for (int t = 0; t < 6; ++t) zc[t] = D[p.o_x0 + 6 * c + t];
    zc[(N - 1) * 8 + 6] = 0.0; zc[(N - 1) * 8 + 7] = 0.0;
    for (int i = 0; i + 1 < N; ++i)
      for (int ax = 0; ax < 2; ++ax) {
        const double P = zc[i * 8 + 3 * ax], V = zc[i * 8 + 3 * ax + 1], A = zc[i * 8 + 3 * ax + 2], U = zc[i * 8 + 6 + ax];
        zc[(i + 1) * 8 + 3 * ax] = P + p.ts * V + p.c2 * A + p.c3 * U;
        zc[(i + 1) * 8 + 3 * ax + 1] = V + p.ts * A + p.c2 * U;
        zc[(i + 1) * 8 + 3 * ax + 2] = A + p.ts * U;
      }
    int jp = I[p.o_initreg + c] - 1;
    jeff_s[c * 64] = jp;
    for (int i = 1; i < N; ++i) {
      const unsigned char m = dec[p.off_mode + c * N + i];
      int j = (m == UNDEC) ? jp : (m == MODE_FROZEN) ? jp : (m >> 2);
      jeff_s[c * 64 + i] = j; jp = j;
    }
  }
  __syncthreads();
  const double vm = p.vm;
  for (int q = tid; q < C * N; q += nt) {
    const int c = q / N, i = q % N;
    const double *y = z + ((long)c * N + i) * 8;
    const int blk[8] = {B_PX, B_VX, B_AX, B_PY, B_VY, B_AY, B_UX, B_UY};
    for (int t = 0; t < 8; ++t) x[col_core(p, blk[t], c, i)] = y[t];
    const int j = jeff_s[c * 64 + i];
    double fxu, fxl, fyu, fyl;
    if (i == 0) {
      fxu = fxl = D[p.o_front0 + 2 * c]; fyu = fyl = D[p.o_front0 + 2 * c + 1];
    } else {
      const double *ft = D + p.o_fronttab + 12 * (c * R + j);
      fxu = y[Y_PX] + (ft[0] + ft[1] * y[Y_VX] + ft[2] * y[Y_VY]);
      fxl = y[Y_PX] + (ft[3] + ft[4] * y[Y_VX] + ft[5] * y[Y_VY]);
      fyu = y[Y_PY] + (ft[6] + ft[7] * y[Y_VX] + ft[8] * y[Y_VY]);
      fyl = y[Y_PY] + (ft[9] + ft[10] * y[Y_VX] + ft[11] * y[Y_VY]);
    }
    x[col_core(p, B_XFU, c, i)] = fxu; x[col_core(p, B_XFL, c, i)] = fxl;
    x[col_core(p, B_YFU, c, i)] = fyu; x[col_core(p, B_YFL, c, i)] = fyl;
    x[col_ar(p, c, i, j)] = 1.0;
    if (i > 0) {
      const unsigned char m = dec[p.off_mode + c * N + i];
      double b[4] = {(y[Y_VX] <= vm) ? 1.0 : 0.0, (y[Y_VY] <= vm) ? 1.0 : 0.0, (y[Y_VX] >= -vm) ? 1.0 : 0.0, (y[Y_VY] >= -vm) ? 1.0 : 0.0};
      double rho = 0.0;
      if (m == MODE_FROZEN) { b[0] = b[1] = b[2] = b[3] = 1.0; rho = 1.0; }
      else b[m & 3] = 0.0;
      for (int t = 0; t < 4; ++t) x[col_rcna(p, t, c, i)] = b[t];
      x[col_rcna(p, 4, c, i)] = rho;
    }
    for (int pt = 0; pt < 5; ++pt) {
      const double PX = (pt == 0) ? y[Y_PX] : ((pt == 1 || pt == 3) ? fxu : fxl);
      const double PY = (pt == 0) ? y[Y_PY] : ((pt == 1 || pt == 2) ? fyu : fyl);
      if (E > 0) {
        int e = (E == 1) ? 0 : dec[p.off_env + (c * N + i) * 5 + pt];
        if (i == 0 && E > 1) {  // nothing is decided at the fixed initial state: pick the containing polygon
          double bestv = -MQ_INF; e = 0;
          for (int ee = 0; ee < E; ++ee) {
            double mn = MQ_INF;
            for (int ed = I[p.o_env_off + ee]; ed < I[p.o_env_off + ee + 1]; ++ed) {
              const double *g = D + p.o_env_edges + 4 * ed;
              mn = fmin(mn, (g[2] - g[0]) * (PY - g[1]) - (PX - g[0]) * (g[3] - g[1]));
            }
            if (mn > bestv) { bestv = mn; e = ee; }
          }
        }
        for (int ee = 0; ee < E; ++ee) x[col_nwe(p, pt, c, ee, i)] = (ee == e) ? 0.0 : 1.0;
      }
      for (int o = 0; o < O; ++o) {
        unsigned char d = dec[p.off_obs + ((c * O + o) * N + i) * 5 + pt];
        const int ne = I[p.o_obs_nedges + o * N + i];
        if (i == 0) {
          double bestv = MQ_INF; d = 0;
          for (int ed = 0; ed < ne; ++ed) {
            const double *g = D + p.o_obs_edges + 4 * ((o * N + i) * L + ed);
            const double cr = (g[2] - g[0]) * (PY - g[1]) - (PX - g[0]) * (g[3] - g[1]);
            if (cr < bestv) { bestv = cr; d = (unsigned char)ed; }
          }
          if (bestv > 1e-9 && I[p.o_obs_soft + o] == 1) d = OBS_SOFT;
        }
        // env point order (UU,LU,UL,LL) -> obstacle front index 4-pt (LL,UL,LU,UU)
        for (int ed = 0; ed < ne; ++ed) {
          const double v = (d == OBS_SOFT || ed != d) ? 1.0 : 0.0;
          if (pt == 0) x[col_dcc(p, c, o, i, ed)] = v; else x[col_dcf(p, c, o, i, ed, 4 - pt)] = v;
        }
        if (d == OBS_SOFT) { if (pt == 0) x[col_so(p, c, o, i)] = 1.0; else x[col_sof(p, c, o, i, 4 - pt)] = 1.0; }
      }
    }
  }
  // collision sides and slacks of every pair (agent_collision_constraints.mod:38-73): the binary of
  // the chosen side is 0, the other three are 1; indices (k1, k2) = (a, b-1), upper triangle
  for (int q = tid; q < p.P * N; q += nt) {
    const int pr = q / N, i = q % N;
    int a = 0, rem = pr;
    while (rem >= C - 1 - a) { rem -= C - 1 - a; ++a; }
    const int b = a + 1 + rem;
    for (int qd = 0; qd < 4; ++qd) {
      unsigned char d = dec[p.off_pair + (pr * N + i) * 4 + qd];
      if (d > 3) d = 0;
      for (int side = 0; side < 4; ++side) x[col_c2c(p, a, b - 1, i, qd * 4 + side)] = (side == d) ? 0.0 : 1.0;
    }
    for (int sq = 0; sq < 4; ++sq) {
      const double v = z[(long)C * N * 8 + (pr * N + i) * 4 + sq];
      x[col_sv(p, a, b - 1, i, sq)] = v > 0.0 ? v : 0.0;
    }
  }
}

// Result of one finished (or stopped) plan s: best bound = smallest bound still open or pruned by the gap rule, into best_bound[s];
// the incumbent's full column vector into xall (zeros without an incumbent) and its exact trajectory in inc_z.  One block of at
// most 128 threads per plan; red: shared [128], jeff_s: shared [8 * 64].  bnb_finish_kernel (end of a run) and
// bnb_harvest_finish_kernel (plans of a streaming run, in the round select marks them finished) run the same code.
__device__ __forceinline__ void finish_plan(const BnbState &st, int s, const DevProb &p, const double *D, const int *I,
                                            double *xall, double *best_bound, double *red, int *jeff_s) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const long pb = (long)s * st.cap;
  double lb = MQ_INF;
  const int nopen = st.open_cnt[s];
  for (int k = tid; k < nopen; k += nt) lb = fmin(lb, st.bound[pb + st.open_idx[pb + k]]);
  red[tid] = lb;
  __syncthreads();
  if (tid == 0) {
    for (int k = 0; k < nt; ++k) lb = fmin(lb, red[k]);
    lb = fmin(lb, st.pruned_lb[s]);
    const double ub = st.ub[s];
    if (st.done[s] && lb == MQ_INF) lb = ub;  // tree exhausted
    if (ub < MQ_INF && lb > ub) lb = ub;
    best_bound[s] = lb;
  }
  const double ub = st.ub[s];
  double *x = xall + p.x_base;
  for (int k = tid; k < p.ncols; k += nt) x[k] = 0.0;
  __syncthreads();
  if (!(ub < MQ_INF) || st.inc_uid[s] == ~0ULL) return;   // no incumbent of its own (ub may come from another rank: frontier sharding)
  expand_solution(p, D, I, st.inc_dec + (long)s * st.ndec_stride, st.inc_z + (long)s * st.zstride, x, jeff_s);
}

__global__ void bnb_finish_kernel(BnbState st, const DevProb *probs, const double *dblob, const int *iblob,
                                  double *xall, double *best_bound) {
  const int s = blockIdx.x;
  __shared__ double red[128];
  __shared__ int jeff_s[8 * 64];
  // streaming run: a plan harvested in an earlier round has its result in place (expand_solution rewrites inc_z: not twice)
  if (st.delivered && st.delivered[s]) return;
  finish_plan(st, s, probs[s], dblob, iblob, xall, best_bound, red, jeff_s);
}

void launch_bnb_finish(const BnbState &st, const DevProb *probs, const double *dblob, const int *iblob,
                       double *xall, double *best_bound, cudaStream_t s) {
  bnb_finish_kernel<<<st.count, 128, 0, s>>>(st, probs, dblob, iblob, xall, best_bound);
}

// solution pool entries of plan k as full column vectors (miqp_b200_pool_fetch); the trajectory is integrated in a copy of the
// stored relaxed optimum, so the pool stays as the search left it
__global__ void pool_expand_kernel(BnbState st, int k, const int *idx, const DevProb *eprobs, const double *dblob, const int *iblob,
                                   double *zs, double *xall) {
  const int e = blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x;
  const DevProb &p = eprobs[e];
  __shared__ int jeff_s[8 * 64];
  const long ent = (long)k * st.pool_cap + idx[e];
  const double *zp = st.pool_z + ent * st.zstride;
  double *z = zs + (long)e * st.zstride;
  double *x = xall + p.x_base;
  for (int q = tid; q < st.zstride; q += nt) z[q] = zp[q];
  for (int q = tid; q < p.ncols; q += nt) x[q] = 0.0;
  __syncthreads();
  expand_solution(p, dblob, iblob, st.pool_dec + ent * st.ndec_stride, z, x, jeff_s);
}

void launch_pool_expand(const BnbState &st, int k, const int *idx, int n, const DevProb *eprobs, const double *dblob, const int *iblob,
                        double *zs, double *xall, cudaStream_t s) {
  if (n > 0) pool_expand_kernel<<<n, 128, 0, s>>>(st, k, idx, eprobs, dblob, iblob, zs, xall);
}

// ---------------------------------------------------------------------------------------
// merge of the solution pools of several ranks (frontier sharding, miqp_b200_pool_merge)
// ---------------------------------------------------------------------------------------
// The pool policy (pool_slot) applied to the union of the ranks' leaves: the pool_cap best entries by key with pairwise different
// decisions.  The ranks' pools suffice: the best leaf of a decision class in the global top pool_cap has fewer than pool_cap
// distinct classes with a better key on its own rank, so it is in that rank's pool.  A greedy scan in key order over the
// candidates of all ranks accepts every entry whose decisions differ from those accepted so far.  Leaves of the ramp-up are in
// every rank's pool (same uid and decisions): the first copy is accepted, the others are duplicates.  Decisions are the plan's
// own ndec_pad bytes: past them, up to the batch's ndec_stride, a node the multi-car kernel makes from its completion (k.imp)
// carries bytes nothing wrote, which differ between ranks.
constexpr int MERGE_THREADS = 256;

__global__ void __launch_bounds__(MERGE_THREADS) pool_merge_kernel(BnbState st, const DevProb *probs, const unsigned char *g, PoolExportLayout lay,
                                                                   int world) {
  __shared__ double val[POOL_MERGE_MAX];
  __shared__ unsigned long long uid[POOL_MERGE_MAX], hsh[POOL_MERGE_MAX];
  __shared__ int src[POOL_MERGE_MAX];
  __shared__ int acc[64];
  __shared__ int nvalid;
  const int k = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  const int cap = st.pool_cap, nw = probs[k].ndec_pad / 16;
  constexpr int NONE = 0x7fffffff;
  // candidate i = entry i % cap of rank i / cap
  auto entry = [=](int i) { return (long)k * cap + i % cap; };
  auto dec_of = [=](int i) {
    return reinterpret_cast<const uint4 *>(g + (long)(i / cap) * lay.bytes + lay.off_dec + entry(i) * st.ndec_stride);
  };
  auto rec_of = [=](int i) { return reinterpret_cast<const PoolRec *>(g + (long)(i / cap) * lay.bytes + lay.off_rec) + entry(i); };
  const int n = world * cap;
  int np = 1;
  while (np < n) np <<= 1;
  if (tid == 0) nvalid = 0;
  for (int i = tid; i < np; i += nt) {
    double v = MQ_INF; unsigned long long u = ~0ULL; int c = NONE;
    if (i < n) {
      const int cnt = reinterpret_cast<const int *>(g + (long)(i / cap) * lay.bytes + lay.off_cnt)[k];
      if (i % cap < min(max(cnt, 0), cap)) { const PoolRec *r = rec_of(i); v = r->val; u = r->uid; c = i; }
    }
    val[i] = v; uid[i] = u; src[i] = c;
  }
  __syncthreads();
  // bitonic sort by (value, uid, candidate index); the empty slots (inf, ~0, NONE) go last
  for (int kk = 2; kk <= np; kk <<= 1)
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < np; i += nt) {
        const int l = i ^ j;
        if (l <= i) continue;
        const bool l_first = pool_key_less(val[l], uid[l], val[i], uid[i]) || (val[l] == val[i] && uid[l] == uid[i] && src[l] < src[i]);
        if (((i & kk) == 0) == l_first) {
          const double tv = val[i]; val[i] = val[l]; val[l] = tv;
          const unsigned long long tu = uid[i]; uid[i] = uid[l]; uid[l] = tu;
          const int tc = src[i]; src[i] = src[l]; src[l] = tc;
        }
      }
      __syncthreads();
    }
  for (int i = tid; i < np; i += nt)
    if (src[i] != NONE && (i + 1 == np || src[i + 1] == NONE)) nvalid = i + 1;
  __syncthreads();
  const int nv = nvalid;
  // 64-bit hash of every candidate's decision bytes (one warp per candidate; a sum, so the order of the lanes does not matter).
  // Only a filter: candidates with equal hashes are compared byte for byte.
  const int lane = tid & 31;
  for (int i = tid >> 5; i < nv; i += nt >> 5) {
    const uint4 *d = dec_of(src[i]);
    unsigned long long h = 0;
    for (int w = lane; w < nw; w += 32) {
      const uint4 q = d[w];
      h += mix64((((unsigned long long)q.y << 32) | q.x) ^ mix64((((unsigned long long)q.w << 32) | q.z) + (unsigned long long)w));
    }
    for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(FULL, h, o);
    if (lane == 0) hsh[i] = h;
  }
  __syncthreads();
  // greedy scan in key order (every branch below depends on shared memory only: uniform over the block)
  int nacc = 0;
  for (int i = 0; i < nv && nacc < cap; ++i) {
    bool dup = false;
    for (int a = 0; a < nacc && !dup; ++a) {
      if (hsh[acc[a]] != hsh[i]) continue;
      const uint4 *x = dec_of(src[acc[a]]), *y = dec_of(src[i]);
      int diff = 0;
      for (int w = tid; w < nw; w += nt) {
        const uint4 p = x[w], q = y[w];
        diff |= (p.x != q.x) || (p.y != q.y) || (p.z != q.z) || (p.w != q.w);
      }
      dup = !__syncthreads_or(diff);
    }
    if (!dup) {
      if (tid == 0) acc[nacc] = i;
      ++nacc;
    }
    __syncthreads();
  }
  // the accepted entries, in key order, into this solver's pool
  const PoolRef pr = pool_ref(st, k);
  for (int a = 0; a < nacc; ++a) {
    const int c = src[acc[a]];
    const double *z = reinterpret_cast<const double *>(g + (long)(c / cap) * lay.bytes + lay.off_z) + entry(c) * st.zstride;
    for (int q = tid; q < st.zstride; q += nt) pr.z[(long)a * st.zstride + q] = z[q];
    const uint4 *d = dec_of(c);
    uint4 *dd = reinterpret_cast<uint4 *>(pr.dec + (long)a * st.ndec_stride);
    for (int w = tid; w < st.ndec_stride / 16; w += nt) dd[w] = d[w];
    if (tid == 0) pr.rec[a] = *rec_of(c);
  }
  if (tid == 0) *pr.cnt = nacc;
}

void launch_pool_merge(const BnbState &st, const DevProb *probs, const unsigned char *gathered, const PoolExportLayout &lay, int world,
                       cudaStream_t s) {
  pool_merge_kernel<<<st.count, MERGE_THREADS, 0, s>>>(st, probs, gathered, lay, world);
}

// ---------------------------------------------------------------------------------------
// streaming runs: harvest of the plans that bnb_select_kernel marked finished, in the same round.  Once select has set done[s],
// nothing of the search writes plan s again, so its result is final.  The host launches the kernels after select and before the
// node kernels, sizing the grids by the plans still active in the previous round (an upper bound of the plans select can finish
// now), at most HARVEST_GRID blocks that stride over the harvested plans: a round that finishes few plans launches few blocks.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SEL_THREADS) bnb_harvest_kernel(BnbState st, int all, int *list, int *n, double *max_viol) {
  __shared__ int warp_tot[SEL_THREADS / 32];
  int base_out = 0;
  for (int base = 0; base < st.count; base += SEL_THREADS) {
    const int s = base + threadIdx.x;
    const int take = (s < st.count && !st.delivered[s] && (all || st.done[s] != 0)) ? 1 : 0;
    int total; const int rank = block_excl_scan(take, warp_tot, total);   // ascending plan order, no atomics: deterministic
    if (take) { list[base_out + rank] = s; st.delivered[s] = 1; max_viol[s] = 0.0; }   // (evaluate_list_kernel takes the maximum into it)
    base_out += total;
  }
  if (threadIdx.x == 0) *n = base_out;
}

__global__ void bnb_harvest_finish_kernel(BnbState st, const DevProb *probs, const double *dblob, const int *iblob, const int *list,
                                          const int *n, double *xall, double *best_bound) {
  __shared__ double red[128];
  __shared__ int jeff_s[8 * 64];
  const int nh = *n;
  for (int e = blockIdx.x; e < nh; e += gridDim.x) {
    const int s = list[e];
    finish_plan(st, s, probs[s], dblob, iblob, xall, best_bound, red, jeff_s);
    __syncthreads();   // red / jeff_s are reused by the next plan
  }
}

__global__ void bnb_harvest_pack_kernel(BnbState st, const DevProb *probs, const int *list, const int *n, const double *obj,
                                        const double *viol, const double *best_bound, double *out, long rec_stride) {
  const int nh = *n;
  for (int e = blockIdx.x; e < nh; e += gridDim.x) {
    const int s = list[e];
    const DevProb &p = probs[s];
    double *rec = out + (long)e * rec_stride;
    if (threadIdx.x == 0) {
      StreamRec r;
      r.objective = obj[s]; r.max_violation = viol[s]; r.best_bound = best_bound[s]; r.ub = st.ub[s];
      r.inc_uid = st.inc_uid[s];
      r.nodes = st.stat_nodes[s]; r.iters = st.stat_iters[s]; r.rows = st.stat_rows[s]; r.uncert = st.stat_uncert[s];
      r.k = s; r.done = st.done[s]; r.done_round = st.done_round[s]; r.overflow = st.overflow[s];
      *reinterpret_cast<StreamRec *>(rec) = r;
    }
    const double *z = st.inc_z + (long)s * st.zstride;
    const int nz = p.C * p.N * 8;
    for (int q = threadIdx.x; q < nz; q += blockDim.x) rec[STREAM_REC_HDR + q] = z[q];
  }
}

void launch_bnb_harvest(const BnbState &st, int all, int *list, int *n, double *max_viol, cudaStream_t s) {
  bnb_harvest_kernel<<<1, SEL_THREADS, 0, s>>>(st, all, list, n, max_viol);
}

void launch_bnb_harvest_finish(const BnbState &st, const DevProb *probs, const double *dblob, const int *iblob, const int *list,
                               const int *n, int max_n, double *xall, double *best_bound, cudaStream_t s) {
  if (max_n > 0) bnb_harvest_finish_kernel<<<(max_n < HARVEST_GRID ? max_n : HARVEST_GRID), 128, 0, s>>>(st, probs, dblob, iblob, list, n, xall, best_bound);
}

void launch_bnb_harvest_pack(const BnbState &st, const DevProb *probs, const int *list, const int *n, int max_n, const double *obj,
                             const double *viol, const double *best_bound, double *out, long rec_stride, cudaStream_t s) {
  if (max_n > 0) bnb_harvest_pack_kernel<<<(max_n < HARVEST_GRID ? max_n : HARVEST_GRID), 128, 0, s>>>(st, probs, list, n, obj, viol, best_bound, out, rec_stride);
}

}  // namespace miqp
