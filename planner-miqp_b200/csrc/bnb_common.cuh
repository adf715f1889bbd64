// bnb_common.cuh -- small device helpers shared by the node kernels (bnb.cu, bnb_multi.cu).
#pragma once
#include "dev_problem.cuh"
#include "kernels.cuh"

namespace miqp {

__device__ __forceinline__ void atomic_min_double(double *addr, double v) {
  unsigned long long *a = reinterpret_cast<unsigned long long *>(addr);
  unsigned long long old = *a;
  while (__longlong_as_double((long long)old) > v) {
    unsigned long long assumed = old;
    old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(v));
    if (old == assumed) break;
  }
}

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
__device__ __forceinline__ void warp_unlock(int *lk, int lane) {   // every lane's writes are fenced before lane 0 releases
  __threadfence();
  __syncwarp();
  if (lane == 0) atomicExch(lk, 0);
  __syncwarp();
}

__device__ __forceinline__ unsigned long long ordered_bits(double v) {
  long long b = __double_as_longlong(v);
  unsigned long long u = (unsigned long long)b;
  return (b < 0) ? ~u : (u | 0x8000000000000000ULL);
}

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
  return x;
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
// held by every thread of the group that holds it (rank in [0, size); any(): group-wide OR, also a barrier of the group).
// Policy: the `cap` best entries by key, distinct decision bytes; a duplicate keeps the better key.  The result depends only on
// the set of leaves offered, not on their order: whatever is evicted or refused has `cap` distinct better entries in the pool.
// Entries other threads of the grid wrote under the lock are read through L2 (__ldcg).
template <class AnyFn>
__device__ __forceinline__ int pool_slot(const PoolRef &pr, const unsigned char *dec, double val, unsigned long long uid, int rank,
                                         int size, AnyFn any) {
  const int cnt = __ldcg(pr.cnt);
  const int nw = pr.ndec_stride / 16;
  const uint4 *mine = reinterpret_cast<const uint4 *>(dec);
  for (int e = 0; e < cnt; ++e) {
    const uint4 *other = reinterpret_cast<const uint4 *>(pr.dec + (long)e * pr.ndec_stride);
    bool diff = false;
    for (int k = rank; k < nw; k += size) {
      const uint4 a = __ldcg(other + k), b = mine[k];
      diff |= (a.x != b.x) || (a.y != b.y) || (a.z != b.z) || (a.w != b.w);
    }
    if (!any(diff)) {   // the same decisions: keep the better key
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

}  // namespace miqp
