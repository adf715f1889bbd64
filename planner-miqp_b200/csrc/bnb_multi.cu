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

long multi_workspace_bytes(int C, int N, int P, int kmax, int ndec_stride) {
  return (multi_layout(C, N, P, kmax, ndec_stride).total_bytes + 15) & ~15L;
}

__global__ void __launch_bounds__(MULTI_MAX_THREADS) bnb_nodes_multi_kernel(BnbState st, const DevProb *probs, const double *dblob,
                                                                            const int *iblob, double *gws, long ws_bytes, int use_smem, int round) {
  extern __shared__ __align__(16) unsigned char smem_multi[];
  __shared__ MShared sh;
  __shared__ int s_word;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const CtaGroup g{tid, nthr, &s_word};
  double *ws = use_smem ? reinterpret_cast<double *>(smem_multi)
                        : reinterpret_cast<double *>(reinterpret_cast<unsigned char *>(gws) + (size_t)blockIdx.x * ws_bytes);
  const int nwork = *reinterpret_cast<volatile int *>(st.work_cnt2);
  MCtx k;
  k.D = dblob; k.I = iblob; k.tid = tid; k.nthr = nthr;

  for (;;) {
    int wi = 0;
    if (tid == 0) wi = atomicAdd(st.work_next2, 1);
    wi = g.bcast(wi);
    if (wi >= nwork) break;
    const int2 item = st.work2[wi];
    const int s = item.x, slot = item.y;
    const DevProb &p = probs[s];
    const long pb = (long)s * st.cap;
    multi_bind(k, &p, ws, st.ndec_stride);
    copy_dec(g, k.dec, st.dec + (pb + slot) * st.ndec_stride, st.ndec_stride);
    const double nbound = st.bound[pb + slot];
    const int2 nmeta = st.meta[pb + slot];
    const unsigned long long nuid = st.uid[pb + slot];
    const double cutoff = st.cutoff[s];
    __syncthreads();

    const MNodeOut out = m_process_node(k, &sh, nbound, cutoff, p.ndec_pad);
    if (tid == 0) count_node(st, s, out.iters, out.rows);
    if (out.what == MN_INFEASIBLE) continue;
    const bool books = (nmeta.x & DEPTH_HEUR) == 0;   // a heuristic completion (below) is never in the bound books
    if (out.what == MN_UNKNOWN) { if (tid == 0 && books) close_uncertified(st, s, nbound); continue; }
    if (out.what == MN_PRUNED) { if (tid == 0 && books) atomic_min_double(&st.pruned_lb[s], out.obj); continue; }
    if (out.what == MN_INCUMBENT) {
      const Traj t = {k.Z, k.nz, k.C, k.N, k.sig + SG_VAL, SG_SIZE, k.P};
      offer_leaf(g, st, s, k.dec, t, out.fval, out.obj, out.converged, books, nuid, round);
      continue;
    }
    // children (those whose lower bound reaches the cutoff were dropped by m_process_node)
    if (tid == 0 && out.pruned_min < MQM_INF) atomic_min_double(&st.pruned_lb[s], out.pruned_min);
    const int nreal = out.nalt;
    if (nreal == 0) continue;
    // Primal heuristic while the plan has no incumbent: the completion of this node by the least violated alternative of every
    // open disjunction (k.imp) goes in as one extra, fully decided node.  It is redundant -- the children still cover the node --
    // so it is flagged (DEPTH_HEUR: never counted in the bounds) and costs one relaxation; with dozens of
    // violated collision disjunctions (8 cars) it finds a first incumbent hundreds of dive levels early.
    const int nheur = (st.multi_heur > 0 && !(cutoff < MQM_INF) && out.soff >= 0 && nmeta.x < DEPTH_MIP_START && (nmeta.x % st.multi_heur) == 0) ? 1 : 0;
    if (tid == 0 && nheur) { sh.alts[nreal] = k.imp[out.soff]; sh.cb[nreal] = out.obj; }   // read by thread 0 only
    push_children(g, st, s, round, nmeta.x, nuid, out.obj, nreal, out.from_imp ? k.imp : k.dec, nheur, k.imp, out.soff, sh.alts, sh.cb,
                  k.imp, nullptr);
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
