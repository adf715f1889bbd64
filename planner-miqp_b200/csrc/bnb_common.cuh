// bnb_common.cuh -- what the two node kernels (bnb.cu: a warp per node, bnb_multi.cu: a CTA per node) do with a solved node,
// written once: the node record encoding, the alternatives of a branching disjunction, the drop of children at the cutoff, the
// incumbent and solution pool update under the plan's lock, and the children.  The part above MQ_EMULATE also compiles for the
// host (the CPU emulation of the multi-car search, tests/emu).
#pragma once
#include "dev_problem.cuh"
#ifndef MQ_EMULATE
#include "kernels.cuh"
#endif

namespace miqp {

// ---- node records (BnbState::meta = (depth word, meta word), BnbState::uid) ----------------------------------------------
// depth word: the depth in the tree, or a flag for the nodes whose depth is not counted
constexpr int DEPTH_MIP_START = 1 << 20;   // the MIP start and its subtree: children keep the word
constexpr int DEPTH_HEUR = 1 << 21;        // heuristic completion (bnb_multi.cu): redundant, never in the bound books
__host__ __device__ __forceinline__ int child_depth(int depth) { return depth >= DEPTH_MIP_START ? depth : depth + 1; }
// meta word: round the node was created in, rank among its siblings (-1: the alternative the parent's completion takes)
__host__ __device__ __forceinline__ int meta_word(int birth, int rank) { return (birth << 8) | (rank + 1); }
__host__ __device__ __forceinline__ int meta_rank(int m) { return (m & 0xff) - 1; }
__host__ __device__ __forceinline__ int meta_birth(int m) { return m >> 8; }

__host__ __device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
  return x;
}
// uid of child a of node `uid` (the root is 1, the MIP start 2)
__host__ __device__ __forceinline__ unsigned long long child_uid(unsigned long long uid, int a) {
  return mix64(uid * 0x9e3779b97f4a7c15ULL + (unsigned long long)(a + 1));
}

// ---- branching ------------------------------------------------------------------------------------------------------------
// Alternatives of the branching disjunction of kind 1 (mode of car c at stage i), 2 (environment polygon of point pt), 3 (edge of
// obstacle o for point pt) or 4 (side of quadruple q of pair pr): sets soff, the byte of the disjunction in a node's decisions, and
// returns the number of alternatives; alts[] gets them when it is not null.
__host__ __device__ __forceinline__ int branch_alts(const DevProb &p, const int *I, int kind, int c, int i, int o, int pt, int pr,
                                                    int q, int &soff, unsigned char *alts) {
  const int N = p.N;
  if (kind == 1) {
    soff = p.off_mode + c * N + i;
    const int na = I[p.o_nalt + c];
    if (alts) { alts[0] = MODE_FROZEN; for (int a = 0; a < na; ++a) alts[1 + a] = (unsigned char)I[p.o_alt + c * 4 * p.R + a]; }
    return na + 1;
  }
  if (kind == 2) {
    soff = p.off_env + (c * N + i) * 5 + pt;
    if (alts) for (int e = 0; e < p.E; ++e) alts[e] = (unsigned char)e;
    return p.E;
  }
  if (kind == 3) {
    soff = p.off_obs + ((c * p.O + o) * N + i) * 5 + pt;
    const int ne = I[p.o_obs_nedges + o * N + i];
    const int soft = I[p.o_obs_soft + o] == 1;
    if (alts) { for (int e = 0; e < ne; ++e) alts[e] = (unsigned char)e; if (soft) alts[ne] = OBS_SOFT; }
    return ne + soft;
  }
  soff = p.off_pair + (pr * N + i) * 4 + q;
  if (alts) for (int e = 0; e < 4; ++e) alts[e] = (unsigned char)e;
  return 4;
}

// Drops the children whose bound cb[a] reaches the cutoff (the others keep their order in alts / cb): returns how many are kept;
// `dropped` is the least bound dropped (+inf if none), which stays in the bound books.
__host__ __device__ __forceinline__ int drop_cut_children(unsigned char *alts, double *cb, int n, double cutoff, double &dropped) {
  int nk = 0;
  dropped = HUGE_VAL;
  for (int a = 0; a < n; ++a) {
    if (cb[a] >= cutoff) { dropped = fmin(dropped, cb[a]); continue; }
    alts[nk] = alts[a]; cb[nk] = cb[a]; ++nk;
  }
  return nk;
}

#ifndef MQ_EMULATE

__device__ __forceinline__ void atomic_min_double(double *addr, double v) {
  unsigned long long *a = reinterpret_cast<unsigned long long *>(addr);
  unsigned long long old = *a;
  while (__longlong_as_double((long long)old) > v) {
    unsigned long long assumed = old;
    old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(v));
    if (old == assumed) break;
  }
}

__device__ __forceinline__ unsigned long long ordered_bits(double v) {
  long long b = __double_as_longlong(v);
  unsigned long long u = (unsigned long long)b;
  return (b < 0) ? ~u : (u | 0x8000000000000000ULL);
}

// ---- thread groups --------------------------------------------------------------------------------------------------------
// The threads that handle one node together: rank in [0, size); sync(): barrier of the group; any(): group-wide OR (also a
// barrier); bcast(v): rank 0's v in every thread.
struct WarpGroup {   // bnb_nodes_kernel: warp 0 of the team
  int rank;
  static constexpr int size = 32;
  __device__ __forceinline__ void sync() const { __syncwarp(); }
  __device__ __forceinline__ bool any(bool p) const { return __any_sync(0xffffffffu, p) != 0; }
  __device__ __forceinline__ int bcast(int v) const { return __shfl_sync(0xffffffffu, v, 0); }
};
struct CtaGroup {    // bnb_nodes_multi_kernel: the whole CTA
  int rank, size;
  int *word;         // shared memory of bcast()
  __device__ __forceinline__ void sync() const { __syncthreads(); }
  __device__ __forceinline__ bool any(bool p) const { return __syncthreads_or(p) != 0; }
  __device__ __forceinline__ int bcast(int v) const {
    if (rank == 0) *word = v;
    __syncthreads();
    v = *word;
    __syncthreads();   // every thread has read the word before the next bcast() writes it
    return v;
  }
};

// Takes the spin lock `lk` for the calling warp: lane 0 tries, the outcome is broadcast, and all 32 lanes loop together until
// it succeeds.  (A single lane spinning on atomicCAS while the other 31 lanes of its warp wait at a warp-collective or a CTA
// barrier produced intermittent "illegal instruction" faults and hangs on sm_100a under contention -- not reproducible under
// compute-sanitizer; profiles/r2a_scheduler_experiments.md.  Keeping the warp converged while it waits removed them.)
__device__ __forceinline__ void warp_lock(int *lk, int lane) {
  unsigned ns = 20;
  for (;;) {
    int got = 0;
    if (lane == 0) got = (atomicCAS(lk, 0, 1) == 0);
    got = __shfl_sync(0xffffffffu, got, 0);
    if (got) break;
    __nanosleep(ns);
    if (ns < 320) ns *= 2;
  }
  __threadfence();
}

// decision bytes of a node (nbytes: a multiple of 16, both ends 16-byte aligned)
template <class G>
__device__ __forceinline__ void copy_dec(const G &g, unsigned char *dst, const unsigned char *src, int nbytes) {
  const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
  uint4 *d4 = reinterpret_cast<uint4 *>(dst);
  for (int k = g.rank; k < nbytes / 16; k += g.size) d4[k] = s4[k];
}

// A relaxed optimum where a node kernel holds it: the stage vector of car c at stage i at z[i * stride + 8c .. + 8], slack q of
// pair-stage e at slack[(4e + q) * slack_stride] (P pairs, none for a single car).
struct Traj { const double *z; int stride, C, N; const double *slack; int slack_stride, P; };

// ... copied into the record layout of inc_z, pool_z and zpool: [C][N][8], then the slacks [P][N][4]
template <class G>
__device__ __forceinline__ void gather_traj(const G &g, double *dst, const Traj &t) {
  for (int e = g.rank; e < t.C * t.N * 8; e += g.size) {
    const int c = e / (t.N * 8), i = (e / 8) % t.N;
    dst[e] = t.z[(long)i * t.stride + 8 * c + e % 8];
  }
  for (int e = g.rank; e < t.P * t.N * 4; e += g.size) dst[(long)t.C * t.N * 8 + e] = t.slack[(long)e * t.slack_stride];
}

// counters of a solved node (one thread)
__device__ __forceinline__ void count_node(const BnbState &st, int s, int iters, long rows) {
  atomicAdd(&st.stat_nodes[s], 1ULL);
  atomicAdd(&st.stat_iters[s], (unsigned long long)iters);
  atomicAdd(&st.stat_rows[s], (unsigned long long)rows);
}

// A node relaxation neither solved nor refuted (one thread): the node is closed, but its bound stays in the books (the plan
// cannot be reported as proven below it) and the event is counted.
__device__ __forceinline__ void close_uncertified(const BnbState &st, int s, double bound) {
  atomic_min_double(&st.pruned_lb[s], bound);
  atomicAdd(&st.stat_uncert[s], 1ULL);
}

// ---- solution pool --------------------------------------------------------------------------------------------------------
__device__ __forceinline__ PoolRef pool_ref(const BnbState &st, int s) {
  PoolRef r;
  r.cap = st.pool_cap; r.zstride = st.zstride; r.ndec_stride = st.ndec_stride;
  r.z = st.pool_z + (long)s * st.pool_cap * st.zstride;
  r.dec = st.pool_dec + (long)s * st.pool_cap * st.ndec_stride;
  r.rec = st.pool_rec + (long)s * st.pool_cap;
  r.cnt = st.pool_cnt + s;
  return r;
}

__device__ __forceinline__ bool pool_key_less(double v1, unsigned long long u1, double v2, unsigned long long u2) {
  return v1 < v2 || (v1 == v2 && u1 < u2);
}

// Slot of a leaf with decisions `dec` and key (val, uid) in its plan's pool, or -1 if it stays out.  Called with the plan's lock
// held by every thread of the group that holds it.
// Policy: the `cap` best entries by key, distinct decision bytes; a duplicate keeps the better key.  The result depends only on
// the set of leaves offered, not on their order: whatever is evicted or refused has `cap` distinct better entries in the pool.
// Entries other threads of the grid wrote under the lock are read through L2 (__ldcg).
template <class G>
__device__ __forceinline__ int pool_slot(const G &g, const PoolRef &pr, const unsigned char *dec, double val, unsigned long long uid) {
  const int cnt = __ldcg(pr.cnt);
  const int nw = pr.ndec_stride / 16;
  const uint4 *mine = reinterpret_cast<const uint4 *>(dec);
  for (int e = 0; e < cnt; ++e) {
    const uint4 *other = reinterpret_cast<const uint4 *>(pr.dec + (long)e * pr.ndec_stride);
    bool diff = false;
    for (int k = g.rank; k < nw; k += g.size) {
      const uint4 a = __ldcg(other + k), b = mine[k];
      diff |= (a.x != b.x) || (a.y != b.y) || (a.z != b.z) || (a.w != b.w);
    }
    if (!g.any(diff)) {   // the same decisions: keep the better key
      const double ev = __ldcg(&pr.rec[e].val);
      const unsigned long long eu = __ldcg(&pr.rec[e].uid);
      return pool_key_less(val, uid, ev, eu) ? e : -1;
    }
  }
  if (cnt < pr.cap) return cnt;
  int worst = 0; double wv = __ldcg(&pr.rec[0].val); unsigned long long wu = __ldcg(&pr.rec[0].uid);
  for (int e = 1; e < cnt; ++e) {
    const double ev = __ldcg(&pr.rec[e].val);
    const unsigned long long eu = __ldcg(&pr.rec[e].uid);
    if (pool_key_less(wv, wu, ev, eu)) { worst = e; wv = ev; wu = eu; }
  }
  return pool_key_less(val, uid, wv, wu) ? worst : -1;
}

// A leaf goes into its plan's pool if it is among the pool's best (pool_slot); called by the group that holds the plan's lock.
// Out of line so that the node kernels keep their register allocation; it runs only at leaves and only when the pool is on.
template <class G>
__device__ __noinline__ void pool_insert(G g, PoolRef pr, const unsigned char *dec, Traj t, double val, unsigned long long uid,
                                         int round, int converged) {
  const int slot = pool_slot(g, pr, dec, val, uid);
  g.sync();   // every thread has read the pool before it changes
  if (slot < 0) return;
  gather_traj(g, pr.z + (long)slot * pr.zstride, t);
  copy_dec(g, pr.dec + (long)slot * pr.ndec_stride, dec, pr.ndec_stride);
  if (g.rank == 0) {
    PoolRec r; r.val = val; r.uid = uid; r.round = round; r.converged = converged;
    pr.rec[slot] = r;
    const int cnt = __ldcg(pr.cnt);
    if (slot == cnt) *pr.cnt = cnt + 1;
  }
}

// ---- what a node leaves behind ----------------------------------------------------------------------------------------------
// A leaf of plan s (every disjunction decided and satisfied) with decisions dec, relaxed optimum t, value val of that point (never
// below obj, the node's bound) and key (val, uid): under the plan's lock it becomes the incumbent if its key is the smallest, and
// it is offered to the solution pool.  A leaf whose relaxation stalled leaves obj in the bound books (its optimum may lie below the
// stalled point, not below obj) if `books` (false: a heuristic completion).
template <class G>
__device__ __forceinline__ void offer_leaf(const G &g, const BnbState &st, int s, const unsigned char *dec, const Traj &t, double val,
                                           double obj, bool converged, bool books, unsigned long long uid, int round) {
  if (g.rank == 0 && !converged && books) atomic_min_double(&st.pruned_lb[s], obj);
  if (g.rank < 32) warp_lock(&st.lock[s], g.rank);   // (in a CTA the other warps wait at the barrier)
  g.sync();
  int better = 0;
  if (g.rank == 0) {
    const double cur = *reinterpret_cast<volatile double *>(&st.ub[s]);
    const unsigned long long cuid = *reinterpret_cast<volatile unsigned long long *>(&st.inc_uid[s]);
    better = val < cur || (val == cur && uid < cuid);
  }
  if (g.bcast(better)) {
    gather_traj(g, st.inc_z + (long)s * st.zstride, t);
    copy_dec(g, st.inc_dec + (long)s * st.ndec_stride, dec, st.ndec_stride);
    __threadfence();   // the incumbent's vector and decisions are visible before its value
    g.sync();
    if (g.rank == 0) { st.ub[s] = val; st.inc_uid[s] = uid; }
  }
  if (st.pool_cap > 0) pool_insert(g, pool_ref(st, s), dec, t, val, uid, round, converged ? 1 : 0);
  __threadfence();   // every thread's writes are visible before rank 0 releases the lock
  g.sync();
  if (g.rank == 0) atomicExch(&st.lock[s], 0);
  g.sync();
}

// The children of a node of plan s (depth word `depth`, uid, bound obj), pushed onto the plan's open list: n children from src,
// child a with byte soff (if >= 0) set to alts[a]; then nx children from xsrc, flagged DEPTH_HEUR.  Child a has bound cb[a] and
// rank -1 if it takes the alternative of the completion imp.  If the plan's node pool cannot hold them, none is made, the overflow
// is flagged and obj stays in the bound books.  warm (if not null): the relaxed optimum the children start their
// interior-point solves from (zpool).
template <class G>
__device__ __forceinline__ void push_children(const G &g, const BnbState &st, int s, int round, int depth, unsigned long long uid,
                                              double obj, int n, const unsigned char *src, int nx, const unsigned char *xsrc, int soff,
                                              const unsigned char *alts, const double *cb, const unsigned char *imp, const Traj *warm) {
  const long pb = (long)s * st.cap;
  const int m = n + nx;
  int fbase = -1, opos = 0;
  if (g.rank == 0) {
    const int old = atomicSub(&st.free_cnt[s], m);
    if (old < m) { atomicAdd(&st.free_cnt[s], m); atomicExch(&st.overflow[s], 1); atomic_min_double(&st.pruned_lb[s], obj); }
    else { fbase = old - m; opos = atomicAdd(&st.open_cnt[s], m); }
  }
  fbase = g.bcast(fbase);
  if (fbase < 0) return;
  opos = g.bcast(opos);
  for (int a = 0; a < m; ++a) {
    const int cs = st.free_stack[pb + fbase + a];
    unsigned char *dst = st.dec + (pb + cs) * st.ndec_stride;
    copy_dec(g, dst, a < n ? src : xsrc, st.ndec_stride);
    if (warm) gather_traj(g, st.zpool + (pb + cs) * (long)st.zp_stride, *warm);
    g.sync();
    if (g.rank == 0) {
      int rank = 0;
      if (soff >= 0) { dst[soff] = alts[a]; rank = (alts[a] == imp[soff]) ? -1 : a; }
      st.bound[pb + cs] = cb[a];
      st.meta[pb + cs] = make_int2(a < n ? child_depth(depth) : depth | DEPTH_HEUR, meta_word(round, rank));
      st.uid[pb + cs] = child_uid(uid, a);
      st.open_idx[pb + opos + a] = cs;
      if (st.susp_slot) st.susp_slot[pb + cs] = -1;
    }
  }
  g.sync();
}

#endif  // MQ_EMULATE

}  // namespace miqp
