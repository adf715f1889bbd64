// bnb_multi.cu -- node kernel of the branch and bound for plans with several cars.
//
// Same role as bnb_nodes_kernel (bnb.cu) with one CTA per node relaxation: persistent CTAs pull
// (plan, node) items from the second work list of the round, solve the joint node QP of all
// cars (node_qp_multi.cuh), scan the relaxed optimum (bnb_multi_core.cuh) and either record an
// incumbent or push the children onto the plan's pool.  The working set of a node (stage
// Hessians, Riccati gains, slack/multiplier of every row) lives in shared memory when it fits
// (2 cars, N=20: 72 kB; 4 cars: 210 kB) and in a per-CTA slice of HBM otherwise.
#include "kernels.cuh"
#include "bnb_common.cuh"
#include "bnb_multi_core.cuh"

namespace miqp {

constexpr int MULTI_MAX_THREADS = 128;

// solution pool: a leaf of bnb_nodes_multi_kernel (whole CTA, plan lock held) goes in if it is among the pool's best (pool_slot).
// Out of line so that the node kernel keeps its register allocation; it runs only at leaves and only when the pool is on.
__device__ __noinline__ void pool_insert_cta(PoolRef pr, const unsigned char *dec, const double *Z, int nz, const double *sig, int C, int N,
                                             int P, double val, unsigned long long uid, int round, int converged) {
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int slot = pool_slot(pr, dec, val, uid, tid, nthr, [](bool p) { return __syncthreads_or(p) != 0; });
  __syncthreads();   // every thread has read the pool before it changes
  if (slot < 0) return;
  double *z = pr.z + (long)slot * pr.zstride;   // the layout of inc_z
  for (int e = tid; e < C * N * 8; e += nthr) {
    const int c = e / (N * 8), i = (e / 8) % N, t = e % 8;
    z[e] = Z[(long)i * nz + 8 * c + t];
  }
  for (int e = tid; e < P * N * 4; e += nthr) z[(long)C * N * 8 + e] = sig[e * SG_SIZE + SG_VAL];
  const uint4 *s4 = reinterpret_cast<const uint4 *>(dec);
  uint4 *d4 = reinterpret_cast<uint4 *>(pr.dec + (long)slot * pr.ndec_stride);
  for (int e = tid; e < pr.ndec_stride / 16; e += nthr) d4[e] = s4[e];
  if (tid == 0) {
    PoolRec r; r.val = val; r.uid = uid; r.round = round; r.converged = converged;
    pr.rec[slot] = r;
    const int cnt = __ldcg(pr.cnt);
    if (slot == cnt) *pr.cnt = cnt + 1;
  }
  __threadfence();
  __syncthreads();
}

long multi_workspace_bytes(int C, int N, int P, int kmax, int ndec_stride) {
  return (multi_layout(C, N, P, kmax, ndec_stride).total_bytes + 15) & ~15L;
}

__global__ void __launch_bounds__(MULTI_MAX_THREADS) bnb_nodes_multi_kernel(BnbState st, const DevProb *probs, const double *dblob,
                                                                            const int *iblob, double *gws, long ws_bytes, int use_smem, int round) {
  extern __shared__ __align__(16) unsigned char smem_multi[];
  __shared__ MShared sh;
  __shared__ int s_i[4];
  const int tid = threadIdx.x, nthr = blockDim.x;
  double *ws = use_smem ? reinterpret_cast<double *>(smem_multi)
                        : reinterpret_cast<double *>(reinterpret_cast<unsigned char *>(gws) + (size_t)blockIdx.x * ws_bytes);
  const int nwork = *reinterpret_cast<volatile int *>(st.work_cnt2);
  MCtx k;
  k.D = dblob; k.I = iblob; k.tid = tid; k.nthr = nthr;

  for (;;) {
    if (tid == 0) s_i[0] = atomicAdd(st.work_next2, 1);
    __syncthreads();
    const int wi = s_i[0];
    __syncthreads();
    if (wi >= nwork) break;
    const int2 item = st.work2[wi];
    const int s = item.x, slot = item.y;
    const DevProb &p = probs[s];
    const long pb = (long)s * st.cap;
    multi_bind(k, &p, ws, st.ndec_stride);
    {
      const uint4 *s4 = reinterpret_cast<const uint4 *>(st.dec + (pb + slot) * st.ndec_stride);
      uint4 *d4 = reinterpret_cast<uint4 *>(k.dec);
      for (int e = tid; e < st.ndec_stride / 16; e += nthr) d4[e] = s4[e];
    }
    const double nbound = st.bound[pb + slot];
    const int2 nmeta = st.meta[pb + slot];
    const unsigned long long nuid = st.uid[pb + slot];
    const double cutoff = st.cutoff[s];
    __syncthreads();

    const MNodeOut out = m_process_node(k, &sh, nbound, cutoff, p.ndec_pad);
    if (tid == 0) {
      atomicAdd(&st.stat_nodes[s], 1ULL);
      atomicAdd(&st.stat_iters[s], (unsigned long long)out.iters);
      atomicAdd(&st.stat_rows[s], (unsigned long long)out.rows);
    }
    if (out.what == MN_INFEASIBLE) continue;
    const bool redundant = (nmeta.x & (1 << 21)) != 0;   // heuristic completion (below): never in the bound books
    if (out.what == MN_UNKNOWN) {   // closed without optimum or certificate: its bound stays in the books
      if (tid == 0 && !redundant) { atomic_min_double(&st.pruned_lb[s], nbound); atomicAdd(&st.stat_uncert[s], 1ULL); }
      continue;
    }
    if (out.what == MN_PRUNED) { if (tid == 0 && !redundant) atomic_min_double(&st.pruned_lb[s], out.obj); continue; }
    if (out.what == MN_INCUMBENT) {
      if (tid < 32) warp_lock(&st.lock[s], tid);   // (warp 0 waits converged; the other warps wait at the barrier below)
      if (tid == 0) {
        if (!out.converged && !redundant) atomic_min_double(&st.pruned_lb[s], out.obj);   // the leaf's optimum may lie below the stalled point, not below obj
        const double cur = *reinterpret_cast<volatile double *>(&st.ub[s]);
        const unsigned long long cuid = *reinterpret_cast<volatile unsigned long long *>(&st.inc_uid[s]);
        s_i[1] = (out.fval < cur || (out.fval == cur && nuid < cuid)) ? 1 : 0;
      }
      __syncthreads();
      if (s_i[1]) {
        double *iz = st.inc_z + (long)s * st.zstride;
        const int C = k.C, N = k.N;
        for (int e = tid; e < C * N * 8; e += nthr) {
          const int c = e / (N * 8), i = (e / 8) % N, t = e % 8;
          iz[e] = k.Z[(long)i * k.nz + 8 * c + t];
        }
        for (int e = tid; e < k.P * N * 4; e += nthr) iz[(long)C * N * 8 + e] = k.sig[e * SG_SIZE + SG_VAL];
        const uint4 *s4 = reinterpret_cast<const uint4 *>(k.dec);
        uint4 *d4 = reinterpret_cast<uint4 *>(st.inc_dec + (long)s * st.ndec_stride);
        for (int e = tid; e < st.ndec_stride / 16; e += nthr) d4[e] = s4[e];
        __threadfence();
      }
      __syncthreads();
      if (st.pool_cap > 0) pool_insert_cta(pool_ref(st, s), k.dec, k.Z, k.nz, k.sig, k.C, k.N, k.P, out.fval, nuid, round, out.converged);
      if (tid == 0) {
        if (s_i[1]) { st.ub[s] = out.fval; st.inc_uid[s] = nuid; }
        __threadfence();
        atomicExch(&st.lock[s], 0);
      }
      __syncthreads();
      continue;
    }
    // children (those whose lower bound reaches the cutoff were dropped by m_process_node)
    if (tid == 0 && out.pruned_min < MQM_INF) atomic_min_double(&st.pruned_lb[s], out.pruned_min);
    const int nreal = out.nalt;
    if (nreal == 0) continue;
    // Primal heuristic while the plan has no incumbent: the completion of this node by the least violated alternative of every
    // open disjunction (k.imp) goes in as one extra, fully decided node.  It is redundant -- the children still cover the node --
    // so it is flagged (depth bit 21: never counted in the bounds) and costs one relaxation; with dozens of
    // violated collision disjunctions (8 cars) it finds a first incumbent hundreds of dive levels early.
    const int nheur = (st.multi_heur > 0 && !(cutoff < MQM_INF) && out.soff >= 0 && nmeta.x < (1 << 20) && (nmeta.x % st.multi_heur) == 0) ? 1 : 0;
    const int nalt = nreal + nheur;
    if (tid == 0) {
      const int old = atomicSub(&st.free_cnt[s], nalt);
      if (old < nalt) {   // node pool of this plan exhausted: the children are dropped, their bound stays in the books
        atomicAdd(&st.free_cnt[s], nalt); atomicExch(&st.overflow[s], 1); atomic_min_double(&st.pruned_lb[s], out.obj); s_i[1] = 0;
      }
      else { s_i[1] = 1; s_i[2] = old - nalt; s_i[3] = atomicAdd(&st.open_cnt[s], nalt); }
    }
    __syncthreads();
    const int ok = s_i[1], fbase = s_i[2], opos = s_i[3];
    if (ok) {
      for (int a = 0; a < nalt; ++a) {
        const bool heur = (a >= nreal);
        const unsigned char *src = (out.from_imp || heur) ? k.imp : k.dec;
        const int cs = st.free_stack[pb + fbase + a];
        unsigned char *dst = st.dec + (pb + cs) * st.ndec_stride;
        const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
        uint4 *d4 = reinterpret_cast<uint4 *>(dst);
        for (int e = tid; e < st.ndec_stride / 16; e += nthr) d4[e] = s4[e];
        __syncthreads();
        if (tid == 0) {
          int rank = 0;
          if (heur) rank = -1;
          else if (out.soff >= 0) { dst[out.soff] = sh.alts[a]; rank = (sh.alts[a] == k.imp[out.soff]) ? -1 : a; }
          st.bound[pb + cs] = heur ? out.obj : sh.cb[a];
          st.meta[pb + cs] = make_int2(heur ? (nmeta.x | (1 << 21)) : (nmeta.x >= (1 << 20)) ? nmeta.x : nmeta.x + 1, (round << 8) | (rank + 1));
          st.uid[pb + cs] = mix64(nuid * 0x9e3779b97f4a7c15ULL + (unsigned long long)(a + 1));
          st.open_idx[pb + opos + a] = cs;
        }
      }
    }
    __syncthreads();
  }
}

int multi_kernel_max_ctas(int smem_bytes, int threads) {
  int nb = 0;
  if (smem_bytes > 0 && cudaFuncSetAttribute(bnb_nodes_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, bnb_nodes_multi_kernel, threads, smem_bytes) != cudaSuccess) { cudaGetLastError(); return 0; }
  return nb;
}

int launch_bnb_nodes_multi(const BnbState &st, const DevProb *probs, const double *dblob, const int *iblob,
                           double *gws, long ws_bytes, int use_smem, int threads, int ctas, int round, cudaStream_t s) {
  bnb_nodes_multi_kernel<<<ctas, threads, use_smem ? (size_t)ws_bytes : 0, s>>>(st, probs, dblob, iblob, gws, ws_bytes, use_smem, round);
  return (int)cudaGetLastError();
}

}  // namespace miqp
