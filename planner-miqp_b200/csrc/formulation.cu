// formulation.cu -- device-side instantiation of the MIQP of cplexmodel/*.mod.
//
// What the reference does with the OPL interpreter (IloOplModel::generate(),
// src/cplex_wrapper.cpp:98, fed by ModelInputDataSource::read,
// src/model_input_data_source.cpp:180-275) is done here by two kernels:
//
//   prepare_tables_kernel  one CTA per plan: derived tables of the formulation (unit edge
//                          normals, normalised per-region rows, front-axle maps, stage
//                          costs) and the row/non-zero index prefixes of the big-M model.
//   rows_kernel<Sink>      ONE THREAD PER ROW of the big-M model, in OPL instantiation
//                          order.  A thread decodes its row index into (family, step, car,
//                          region/edge/pair, sub-row) in closed form and streams the row
//                          into a sink: CsrSink writes rowptr/lo/hi/cols/vals (adjacent
//                          threads write adjacent segments: coalesced, HBM-write bound),
//                          EvalSink accumulates the row activity of a candidate vector and
//                          its violation (used to certify every incumbent on the device).
//
// This file is compiled with --fmad=false: coefficients are compared bit for bit with the
// CPU oracle (oracle/miqp_oracle.c, built with -ffp-contract=off).
#include "dev_problem.cuh"
#include "kernels.cuh"
#include "formulation_tables.cuh"

namespace miqp {

// ------------------------------------------------------------------------------------------
// prepare_tables_kernel
// ------------------------------------------------------------------------------------------
__global__ void prepare_tables_kernel(DevProb *probs, double *dblob, int *iblob, int count) {
  const int s = blockIdx.x;
  if (s >= count) return;
  DevProb &p = probs[s];
  prepare_tables_parallel(p, dblob, iblob, threadIdx.x, blockDim.x);
  __syncthreads();
  if (threadIdx.x == 0) prepare_tables_serial(p, dblob, iblob);
}

// ------------------------------------------------------------------------------------------
// row emitter
// ------------------------------------------------------------------------------------------
#define INF_D (__longlong_as_double(0x7ff0000000000000LL))

// Sink concept:  void begin(double lo, double hi, long nnz_start);  void add(int col, double val);  void end();
template <class Sink>
__device__ __forceinline__ void emit_row(const DevProb &p, const double *__restrict__ D,
                                         const int *__restrict__ I, long r, Sink &s) {
  const int N = p.N, R = p.R, C = p.C, O = p.O, L = p.L, E = p.E;
  int fam = 0;
  while (fam + 1 < NUM_FAM && r >= p.fam_row[fam + 1]) ++fam;
  const long q = r - p.fam_row[fam];
  const long nz0 = p.fam_nnz[fam];
  switch (fam) {
    case FAM_IC1: {
      int c = (int)(q / 12), k = (int)(q % 12);
      double v; int col;
      if (k < 6) {
        const int blk[6] = {B_PX, B_VX, B_AX, B_PY, B_VY, B_AY};
        v = D[p.o_x0 + 6 * c + k]; col = col_core(p, blk[k], c, 0);
      } else if (k < 10) {
        const int blk[4] = {B_XFU, B_XFL, B_YFU, B_YFL};
        v = D[p.o_front0 + 2 * c + ((k - 6) >> 1)]; col = col_core(p, blk[k - 6], c, 0);
      } else {
        v = 0.0; col = col_core(p, k == 10 ? B_UX : B_UY, c, N - 1);
      }
      s.begin(v, v, nz0 + q); s.add(col, 1.0); s.end();
    } break;
    case FAM_IC2: {
      long idx = q / 5; int k = (int)(q % 5);
      int j = (int)(idx / C), c = (int)(idx % C);
      const int pre[5] = {0, 1, 3, 5, 7};
      int ar = col_ar(p, c, 0, j);
      long nz = nz0 + 9 * idx + pre[k];
      if (k == 0) {
        double on = (j + 1 == I[p.o_initreg + c]) ? 1.0 : 0.0;
        s.begin(on, on, nz); s.add(ar, 1.0); s.end();
      } else {
        int ucol = col_core(p, (k <= 2) ? B_UX : B_UY, c, 0);
        // k=1: ux <= max_jerk_x + M(1-ar); k=2: ux >= min_jerk_x - M(1-ar); k=3,4 same for y
        int limidx = (k == 1) ? 5 : (k == 2) ? 4 : (k == 3) ? 7 : 6;
        double lim = D[p.o_lim[limidx] + c * R + j];
        if (k & 1) { s.begin(-INF_D, lim + BIGM_JERK, nz); s.add(ucol, 1.0); s.add(ar, BIGM_JERK); }
        else { s.begin(lim - BIGM_JERK, INF_D, nz); s.add(ucol, 1.0); s.add(ar, -BIGM_JERK); }
        s.end();
      }
    } break;
    case FAM_IC3: {
      int c = (int)(q / 5), k = (int)(q % 5);
      s.begin(0.0, 0.0, nz0 + q); s.add(col_rcna(p, k, c, 0), 1.0); s.end();
    } break;
    case FAM_DYN: {
      long idx = q / 3; int k = (int)(q % 3);
      int ax = (int)(idx % 2), c = (int)((idx / 2) % C), i = 1 + (int)(idx / (2 * C));
      const int pre[3] = {0, 5, 9};
      int Pb = ax ? B_PY : B_PX, Vb = ax ? B_VY : B_VX, Ab = ax ? B_AY : B_AX, Ub = ax ? B_UY : B_UX;
      s.begin(0.0, 0.0, nz0 + 12 * idx + pre[k]);
      if (k == 0) {
        s.add(col_core(p, Pb, c, i), 1.0); s.add(col_core(p, Pb, c, i - 1), -1.0);
        s.add(col_core(p, Vb, c, i - 1), -p.ts); s.add(col_core(p, Ab, c, i - 1), -p.c2);
        s.add(col_core(p, Ub, c, i - 1), -p.c3);
      } else if (k == 1) {
        s.add(col_core(p, Vb, c, i), 1.0); s.add(col_core(p, Vb, c, i - 1), -1.0);
        s.add(col_core(p, Ab, c, i - 1), -p.ts); s.add(col_core(p, Ub, c, i - 1), -p.c2);
      } else {
        s.add(col_core(p, Ab, c, i), 1.0); s.add(col_core(p, Ab, c, i - 1), -1.0);
        s.add(col_core(p, Ub, c, i - 1), -p.ts);
      }
      s.end();
    } break;
    case FAM_BOX: {
      long idx = q / 12; int k = (int)(q % 12);
      int c = (int)(idx % C), i = (int)(idx / C);
      // vel_y has no upper bound and vel_x two (model_region_constraints.mod:26-27)
      const int blk[12] = {B_VX, B_VY, B_VX, B_VX, B_AX, B_AX, B_AY, B_AY, B_UX, B_UX, B_UY, B_UY};
      double lo = -INF_D, hi = INF_D;
      switch (k) {
        case 0: case 1: lo = p.min_vel; break;
        case 2: case 3: hi = p.max_vel; break;
        case 4: case 6: hi = p.total_max_acc; break;
        case 5: case 7: lo = p.total_min_acc; break;
        case 8: case 10: hi = p.total_max_jerk; break;
        default: lo = p.total_min_jerk; break;
      }
      s.begin(lo, hi, nz0 + q); s.add(col_core(p, blk[k], c, i), 1.0); s.end();
    } break;
    case FAM_REGION: {
      const long rps = p.region_rows_car[C];
      int i = 1 + (int)(q / rps);
      long rq = q % rps;
      int c = 0;
      while (c + 1 < C && rq >= p.region_rows_car[c + 1]) ++c;
      rq -= p.region_rows_car[c];
      long nz = nz0 + (long)(i - 1) * p.region_nnz_car[C] + p.region_nnz_car[c];
      const int *pp = I + p.o_posspre + c * (R + 1);
      const int rp = pp[R];
      const long total = 20L * rp + (R - rp) + 1;
      if (rq == total - 1) {  // sum_j active_region = 1  (:113)
        s.begin(1.0, 1.0, nz + 76L * rp + (R - rp));
        for (int j = 0; j < R; ++j) s.add(col_ar(p, c, i, j), 1.0);
        s.end();
        break;
      }
      int lo_j = 0, hi_j = R - 1;  // largest j with j + 19*pp[j] <= rq
      while (lo_j < hi_j) {
        int mid = (lo_j + hi_j + 1) >> 1;
        if ((long)mid + 19L * pp[mid] <= rq) lo_j = mid; else hi_j = mid - 1;
      }
      const int j = lo_j;
      const int k = (int)(rq - ((long)j + 19L * pp[j]));
      nz += 76L * pp[j] + (j - pp[j]);
      const int ar = col_ar(p, c, i, j);
      if (I[p.o_possible + c * R + j] != 1) {  // :108
        s.begin(0.0, 0.0, nz); s.add(ar, 1.0); s.end();
        break;
      }
      const int pre[20] = {0, 4, 8, 13, 18, 23, 28, 33, 38, 43, 48, 50, 52, 54, 56, 58, 60, 62, 64, 70};
      nz += pre[k];
      const double *f = D + p.o_frac + 4 * j;
      const int vx = col_core(p, B_VX, c, i), vy = col_core(p, B_VY, c, i);
      const int rho = col_rcna(p, 4, c, i);
      if (k == 0) {         // :53 wedge
        s.begin(-BIGM_FRAC, INF_D, nz);
        s.add(vy, f[0]); s.add(vx, -f[1]); s.add(ar, -BIGM_FRAC); s.add(rho, BIGM_FRAC); s.end();
      } else if (k == 1) {  // :54
        s.begin(-INF_D, BIGM_FRAC, nz);
        s.add(vy, f[2]); s.add(vx, -f[3]); s.add(ar, BIGM_FRAC); s.add(rho, -BIGM_FRAC); s.end();
      } else if (k < 10) {  // :57-70 front axle box, q4 = x UB, x LB, y UB, y LB; lower then upper row
        int q4 = (k - 2) >> 1, upper = (k - 2) & 1;
        const int polyidx[4] = {2, 3, 0, 1};
        const int fblk[4] = {B_XFU, B_XFL, B_YFU, B_YFL};
        const double *P = D + p.o_poly[polyidx[q4]] + 3 * j;
        const double wb = D[p.o_wb + c];
        if (!upper) s.begin(wb * P[0] - BIGM_FRONT, INF_D, nz); else s.begin(-INF_D, wb * P[0] + BIGM_FRONT, nz);
        s.add(col_core(p, fblk[q4], c, i), 1.0);
        s.add(col_core(p, (q4 < 2) ? B_PX : B_PY, c, i), -1.0);
        s.add(vx, -(wb * P[1])); s.add(vy, -(wb * P[2]));
        s.add(ar, upper ? BIGM_FRONT : -BIGM_FRONT);
        s.end();
      } else if (k < 18) {  // :73-94 jerk then acc boxes: max_x, min_x, max_y, min_y
        int kk = k - 10, isacc = kk >> 2, sub = kk & 3;
        const int limidx_j[4] = {5, 4, 7, 6}, limidx_a[4] = {1, 0, 3, 2};
        double lim = D[p.o_lim[isacc ? limidx_a[sub] : limidx_j[sub]] + c * R + j];
        const double M = isacc ? BIGM_ACC : BIGM_JERK;
        int blk = isacc ? ((sub < 2) ? B_AX : B_AY) : ((sub < 2) ? B_UX : B_UY);
        int vcol = col_core(p, blk, c, i);
        if ((sub & 1) == 0) { s.begin(-INF_D, lim + M, nz); s.add(vcol, 1.0); s.add(ar, M); }
        else { s.begin(lim - M, INF_D, nz); s.add(vcol, 1.0); s.add(ar, -M); }
        s.end();
      } else {              // :97-104 curvature
        const double sl = (f[1] + f[3]) / (f[0] + f[2]);
        const double *KK = D + p.o_poly[k == 18 ? 4 : 5] + 3 * j;
        if (k == 18) s.begin(-INF_D, KK[0] + BIGM_KAPPA, nz); else s.begin(KK[0] - BIGM_KAPPA, INF_D, nz);
        s.add(col_core(p, B_AY, c, i), 1.0); s.add(vx, -KK[1]); s.add(vy, -KK[2]);
        s.add(col_core(p, B_AX, c, i), -sl);
        s.add(ar, k == 18 ? BIGM_KAPPA : -BIGM_KAPPA); s.add(rho, k == 18 ? -BIGM_KAPPA : BIGM_KAPPA);
        s.end();
      }
    } break;
    case FAM_MINSPEED: {
      long idx = q / 15; int k = (int)(q % 15);
      int j = (int)(idx % R), c = (int)((idx / R) % C), i = 1 + (int)(idx / ((long)R * C));
      const int pre[15] = {0, 2, 4, 6, 8, 10, 12, 14, 16, 19, 22, 24, 26, 28, 30};
      long nz = nz0 + 35 * idx + pre[k];
      const double vm = p.vm;
      const int rho = col_rcna(p, 4, c, i);
      if (k < 8) {
        int isy = k >> 2, sub = k & 3;
        int v = col_core(p, isy ? B_VY : B_VX, c, i);
        int bpos = col_rcna(p, isy ? 1 : 0, c, i), bneg = col_rcna(p, isy ? 3 : 2, c, i);
        switch (sub) {
          case 0: s.begin(vm, INF_D, nz); s.add(v, 1.0); s.add(bpos, BIGM_VEL); break;
          case 1: s.begin(-INF_D, vm + BIGM_VEL, nz); s.add(v, 1.0); s.add(bpos, BIGM_VEL); break;
          case 2: s.begin(-INF_D, vm + BIGM_VEL, nz); s.add(v, -1.0); s.add(bneg, BIGM_VEL); break;
          default: s.begin(vm, INF_D, nz); s.add(v, -1.0); s.add(bneg, BIGM_VEL); break;
        }
        s.end();
      } else if (k < 10) {
        if (k == 8) s.begin(-INF_D, 1.0, nz); else s.begin(-1.0, INF_D, nz);
        s.add(col_ar(p, c, i, j), 1.0); s.add(col_ar(p, c, i - 1, j), -1.0); s.add(rho, k == 8 ? 1.0 : -1.0);
        s.end();
      } else if (k < 14) {
        const int order[4] = {0, 1, 2, 3};  // bxp, byp, bxn, byn
        s.begin(-INF_D, 0.0, nz); s.add(rho, 1.0); s.add(col_rcna(p, order[k - 10], c, i), -1.0); s.end();
      } else {
        s.begin(-3.0, INF_D, nz); s.add(rho, 1.0);
        for (int t = 0; t < 4; ++t) s.add(col_rcna(p, t, c, i), -1.0);
        s.end();
      }
    } break;
    case FAM_ENV: {
      const int nE = p.nEnvEdges;
      const long rows = 5L * nE + 5;
      long idx = q / rows; int k = (int)(q % rows);
      int c = (int)(idx % C), i = (int)(idx / C);
      long nz = nz0 + idx * (15L * nE + 5L * E);
      if (k < 5 * nE) {
        int ed = k / 5, pt = k % 5;
        int e = 0;
        while (e + 1 < E && ed >= I[p.o_env_off + e + 1]) ++e;
        const double *g = D + p.o_env_edges + 4 * ed;
        double dx = g[2] - g[0], dy = g[3] - g[1];
        double rhs = dx * g[1] - g[0] * dy;
        // points: rear, (xU,yU), (xL,yU), (xU,yL), (xL,yL)  (obstacle_environment_constraints.mod:17-27)
        const int Xb[5] = {B_PX, B_XFU, B_XFL, B_XFU, B_XFL};
        const int Yb[5] = {B_PY, B_YFU, B_YFU, B_YFL, B_YFL};
        s.begin(rhs, INF_D, nz + 3L * k);
        s.add(col_core(p, Yb[pt], c, i), dx); s.add(col_core(p, Xb[pt], c, i), -dy);
        s.add(col_nwe(p, pt, c, e, i), BIGM_ENV);
        s.end();
      } else {
        int kk = k - 5 * nE;
        s.begin(-INF_D, (double)(E - 1), nz + 15L * nE + (long)kk * E);
        for (int e = 0; e < E; ++e) s.add(col_nwe(p, kk, c, e, i), 1.0);
        s.end();
      }
    } break;
    case FAM_OBS: {
      const int *sr = I + p.o_obsstep_rows;
      int lo_i = 0, hi_i = N - 1;  // largest i with sr[i] <= q
      while (lo_i < hi_i) { int mid = (lo_i + hi_i + 1) >> 1; if ((long)sr[mid] <= q) lo_i = mid; else hi_i = mid - 1; }
      const int i = lo_i;
      long rq = q - sr[i];
      const int *rpre = I + p.o_obsrowpre + i * (O + 1), *npre = I + p.o_obsnnzpre + i * (O + 1);
      int c = (int)(rq / rpre[O]);
      rq -= (long)c * rpre[O];
      int o = 0;
      while (o + 1 < O && rq >= rpre[o + 1]) ++o;
      int k = (int)(rq - rpre[o]);
      long nz = nz0 + I[p.o_obsstep_nnz + i] + (long)c * npre[O] + npre[o];
      const int ne = I[p.o_obs_nedges + o * N + i];
      // points: rear, (xL,yL), (xU,yL), (xL,yU), (xU,yU)  (obstacle_environment_constraints.mod:61-65)
      if (k < 5 * ne) {
        int ed = k / 5, pt = k % 5;
        const double *g = D + p.o_obs_edges + 4 * ((o * N + i) * L + ed);
        double dx = g[2] - g[0], dy = g[3] - g[1];
        double rhs = dx * g[1] - g[0] * dy;
        const int Xb[5] = {B_PX, B_XFL, B_XFU, B_XFL, B_XFU};
        const int Yb[5] = {B_PY, B_YFL, B_YFL, B_YFU, B_YFU};
        int dcol = (pt == 0) ? col_dcc(p, c, o, i, ed) : col_dcf(p, c, o, i, ed, pt - 1);
        s.begin(-INF_D, rhs, nz + 3L * k);
        s.add(col_core(p, Yb[pt], c, i), dx); s.add(col_core(p, Xb[pt], c, i), -dy); s.add(dcol, -BIGM_OBS);
        s.end();
      } else {
        int kk = k - 5 * ne;
        int soft = (I[p.o_obs_soft + o] == 1);
        s.begin(-INF_D, (double)(ne - 1), nz + 15L * ne + (long)kk * (ne + soft));
        for (int ed = 0; ed < ne; ++ed) s.add((kk == 0) ? col_dcc(p, c, o, i, ed) : col_dcf(p, c, o, i, ed, kk - 1), 1.0);
        if (soft) s.add((kk == 0) ? col_so(p, c, o, i) : col_sof(p, c, o, i, kk - 1), -1.0);
        s.end();
      }
    } break;
    case FAM_A2A_ZERO: {
      const int K = p.K;
      long Z = (long)K * (K - 1) / 2;
      long idx = q / 20; int k = (int)(q % 20);
      int i = (int)(idx / Z), z = (int)(idx % Z);
      int k1 = 1;
      while (z >= k1) { z -= k1; ++k1; }
      int k2 = z;
      s.begin(0.0, 0.0, nz0 + q);
      s.add(k < 4 ? col_sv(p, k1, k2, i, k) : col_c2c(p, k1, k2, i, k - 4), 1.0);
      s.end();
    } break;
    default: {  // FAM_A2A
      const int P = p.P;
      long idx = q / 24; int k = (int)(q % 24);
      int i = (int)(idx / P), pr = (int)(idx % P);
      int a = 0, rem = pr;
      while (rem >= C - 1 - a) { rem -= C - 1 - a; ++a; }
      int b = a + 1 + rem;
      const int k1 = a, k2 = b - 1;
      const int pre[24] = {0, 4, 8, 12, 16, 20, 21, 22, 25, 28, 31, 34, 38, 41, 44, 47, 50, 54, 58, 62, 66, 70, 74, 75};
      long nz = nz0 + 76 * idx + pre[k];
      const double RR = D[p.o_radius + a] + D[p.o_radius + b];  // initialization.mod:16-22
      const double saf = D[p.o_safety + i], sls = D[p.o_safety_slack + i];
      const double Dd = RR + saf;
      const double Ds = RR + saf + sls;
#define CC(blk, car) col_core(p, blk, car, i)
#define BB(n) col_c2c(p, k1, k2, i, (n) - 1)
#define SS(n) col_sv(p, k1, k2, i, (n) - 1)
      switch (k) {
        // :41-47 rear/rear
        case 0: s.begin(-INF_D, -Ds, nz); s.add(CC(B_PX, a), 1.0); s.add(CC(B_PX, b), -1.0); s.add(SS(1), -1.0); s.add(BB(1), -BIGM_AGENTS); break;
        case 1: s.begin(Ds, INF_D, nz); s.add(CC(B_PX, a), 1.0); s.add(CC(B_PX, b), -1.0); s.add(SS(1), 1.0); s.add(BB(2), BIGM_AGENTS); break;
        case 2: s.begin(-INF_D, -Ds, nz); s.add(CC(B_PY, a), 1.0); s.add(CC(B_PY, b), -1.0); s.add(SS(2), -1.0); s.add(BB(3), -BIGM_AGENTS); break;
        case 3: s.begin(Ds, INF_D, nz); s.add(CC(B_PY, a), 1.0); s.add(CC(B_PY, b), -1.0); s.add(SS(2), 1.0); s.add(BB(4), BIGM_AGENTS); break;
        case 4: s.begin(-INF_D, 3.0, nz); for (int t = 1; t <= 4; ++t) s.add(BB(t), 1.0); break;
        case 5: s.begin(-INF_D, sls, nz); s.add(SS(1), 1.0); break;
        case 6: s.begin(-INF_D, sls, nz); s.add(SS(2), 1.0); break;
        // :50-54 rear a vs front b
        case 7: s.begin(-INF_D, -Dd, nz); s.add(CC(B_PX, a), 1.0); s.add(CC(B_XFL, b), -1.0); s.add(BB(5), -BIGM_AGENTS); break;
        case 8: s.begin(Dd, INF_D, nz); s.add(CC(B_PX, a), 1.0); s.add(CC(B_XFU, b), -1.0); s.add(BB(6), BIGM_AGENTS); break;
        case 9: s.begin(-INF_D, -Dd, nz); s.add(CC(B_PY, a), 1.0); s.add(CC(B_YFL, b), -1.0); s.add(BB(7), -BIGM_AGENTS); break;
        case 10: s.begin(Dd, INF_D, nz); s.add(CC(B_PY, a), 1.0); s.add(CC(B_YFU, b), -1.0); s.add(BB(8), BIGM_AGENTS); break;
        case 11: s.begin(-INF_D, 3.0, nz); for (int t = 5; t <= 8; ++t) s.add(BB(t), 1.0); break;
        // :57-61 rear b vs front a
        case 12: s.begin(-INF_D, -Dd, nz); s.add(CC(B_PX, b), 1.0); s.add(CC(B_XFL, a), -1.0); s.add(BB(9), -BIGM_AGENTS); break;
        case 13: s.begin(Dd, INF_D, nz); s.add(CC(B_PX, b), 1.0); s.add(CC(B_XFU, a), -1.0); s.add(BB(10), BIGM_AGENTS); break;
        case 14: s.begin(-INF_D, -Dd, nz); s.add(CC(B_PY, b), 1.0); s.add(CC(B_YFL, a), -1.0); s.add(BB(11), -BIGM_AGENTS); break;
        case 15: s.begin(Dd, INF_D, nz); s.add(CC(B_PY, b), 1.0); s.add(CC(B_YFU, a), -1.0); s.add(BB(12), BIGM_AGENTS); break;
        case 16: s.begin(-INF_D, 3.0, nz); for (int t = 9; t <= 12; ++t) s.add(BB(t), 1.0); break;
        // :65-71 front/front
        case 17: s.begin(Ds, INF_D, nz); s.add(CC(B_XFL, a), 1.0); s.add(CC(B_XFU, b), -1.0); s.add(SS(3), 1.0); s.add(BB(13), BIGM_AGENTS); break;
        case 18: s.begin(-INF_D, -Ds, nz); s.add(CC(B_XFU, a), 1.0); s.add(CC(B_XFL, b), -1.0); s.add(SS(3), -1.0); s.add(BB(14), -BIGM_AGENTS); break;
        case 19: s.begin(Ds, INF_D, nz); s.add(CC(B_YFL, a), 1.0); s.add(CC(B_YFU, b), -1.0); s.add(SS(4), 1.0); s.add(BB(15), BIGM_AGENTS); break;
        case 20: s.begin(-INF_D, -Ds, nz); s.add(CC(B_YFU, a), 1.0); s.add(CC(B_YFL, b), -1.0); s.add(SS(4), -1.0); s.add(BB(16), -BIGM_AGENTS); break;
        case 21: s.begin(-INF_D, 3.0, nz); for (int t = 13; t <= 16; ++t) s.add(BB(t), 1.0); break;
        case 22: s.begin(-INF_D, sls, nz); s.add(SS(3), 1.0); break;
        default: s.begin(-INF_D, sls, nz); s.add(SS(4), 1.0); break;
      }
      s.end();
#undef CC
#undef BB
#undef SS
    } break;
  }
}

// ------------------------------------------------------------------------------------------
// sinks
// ------------------------------------------------------------------------------------------
struct CsrSink {
  long *rowptr; int *cols; double *vals; double *lo; double *hi;
  long row;        // global row index in the batch arrays
  long nnz_base;   // plan's base in cols/vals
  long pos;
  int nonzeros;
  __device__ __forceinline__ void begin(double l, double h, long nz) {
    pos = nnz_base + nz;
    if (rowptr) rowptr[row] = pos;
    if (lo) lo[row] = l;
    if (hi) hi[row] = h;
  }
  __device__ __forceinline__ void add(int col, double v) {
    if (cols) cols[pos] = col;
    if (vals) vals[pos] = v;
    nonzeros += (v != 0.0);
    ++pos;
  }
  __device__ __forceinline__ void end() {}
};

struct EvalSink {
  const double *x;
  double lo, hi, act, viol;
  __device__ __forceinline__ void begin(double l, double h, long) { lo = l; hi = h; act = 0.0; }
  __device__ __forceinline__ void add(int col, double v) { act += v * x[col]; }
  __device__ __forceinline__ void end() {
    double v = 0.0;
    if (lo - act > v) v = lo - act;
    if (act - hi > v) v = act - hi;
    if (!(act == act)) v = INF_D;
    viol = v;
  }
};

// grid: x over rows (grid-stride), y over plans
__global__ void assemble_rows_kernel(const DevProb *probs, const double *dblob, const int *iblob, int count,
                                     long *rowptr, int *cols, double *vals, double *lo, double *hi,
                                     unsigned long long *nnz_count /* [count] */) {
  const int s = blockIdx.y;
  if (s >= count) return;
  const DevProb &p = probs[s];
  const long nrows = p.fam_row[NUM_FAM];
  int local = 0;
  for (long r = (long)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (long)gridDim.x * blockDim.x) {
    CsrSink sink{rowptr, cols, vals, lo, hi, p.row_base + s + r, p.nnz_base, 0, 0};
    emit_row(p, dblob, iblob, r, sink);
    local += sink.nonzeros;
  }
  // plan's closing rowptr entry (each plan owns nrows+1 rowptr entries: row_base + s)
  if (blockIdx.x == 0 && threadIdx.x == 0 && rowptr) rowptr[p.row_base + s + nrows] = p.nnz_base + p.fam_nnz[NUM_FAM];
  for (int off = 16; off > 0; off >>= 1) local += __shfl_down_sync(0xffffffffu, local, off);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(&nnz_count[s], (unsigned long long)local);
}

__device__ __forceinline__ void atomic_max_double(double *addr, double v) {
  // v >= 0: IEEE ordering equals unsigned integer ordering
  atomicMax(reinterpret_cast<unsigned long long *>(addr), (unsigned long long)__double_as_longlong(v));
}

// max violation of rows, column bounds and integrality; objective (objective_function.mod:7-19) of plan s: blocks (x, *) of the
// grid share its rows and columns.  evaluate_kernel (every plan) and evaluate_list_kernel (the plans of a list) run the same code,
// so both give the same bits.
__device__ __forceinline__ void evaluate_plan(const DevProb *probs, const double *dblob, const int *iblob, int s,
                                              const double *xall, double *max_viol, double *objective) {
  const DevProb &p = probs[s];
  const double *x = xall + p.x_base;
  const long nrows = p.fam_row[NUM_FAM];
  double worst = 0.0;
  for (long r = (long)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (long)gridDim.x * blockDim.x) {
    EvalSink sink{x, 0, 0, 0, 0};
    emit_row(p, dblob, iblob, r, sink);
    if (sink.viol > worst) worst = sink.viol;
  }
  for (long k = (long)blockIdx.x * blockDim.x + threadIdx.x; k < p.ncols; k += (long)gridDim.x * blockDim.x) {
    bool bin = (k >= p.base_nwe && k < p.base_so) || (k >= p.base_c2c && k < p.base_sv);
    double lo = -INF_D, hi = INF_D;
    if (bin) { lo = 0.0; hi = 1.0; }
    else if (k >= p.base_so && k < p.base_c2c) { lo = 0.0; hi = 1.0; }  // decision_variables.mod:46-47
    else if (k >= p.base_sv) { lo = 0.0; hi = p.maximum_slack; }        // :53
    double xv = x[k], v = 0.0;
    if (lo - xv > v) v = lo - xv;
    if (xv - hi > v) v = xv - hi;
    if (bin) { double rr = fabs(xv - floor(xv + 0.5)); if (rr > v) v = rr; }
    if (!(xv == xv)) v = INF_D;
    if (v > worst) worst = v;
  }
  for (int off = 16; off > 0; off >>= 1) { double o = __shfl_down_sync(0xffffffffu, worst, off); if (o > worst) worst = o; }
  if ((threadIdx.x & 31) == 0 && worst > 0.0) atomic_max_double(&max_viol[s], worst);
  // objective: one thread per plan, same summation order as the oracle (deterministic)
  if (blockIdx.x == 0 && threadIdx.x == 0 && objective) {
    const double *D = dblob;
    const int N = p.N, C = p.C, O = p.O, K = p.K;
    double cost = 0.0;
    for (int i = 0; i < N; ++i)
      for (int c = 0; c < C; ++c) {
        double dpx = x[col_core(p, B_PX, c, i)] - D[p.o_ref[0] + c * N + i];
        double dvx = x[col_core(p, B_VX, c, i)] - D[p.o_ref[1] + c * N + i];
        double dpy = x[col_core(p, B_PY, c, i)] - D[p.o_ref[2] + c * N + i];
        double dvy = x[col_core(p, B_VY, c, i)] - D[p.o_ref[3] + c * N + i];
        double ax = x[col_core(p, B_AX, c, i)], ay = x[col_core(p, B_AY, c, i)];
        double ux = x[col_core(p, B_UX, c, i)], uy = x[col_core(p, B_UY, c, i)];
        cost += D[p.o_w[0] + c] * dpx * dpx + D[p.o_w[1] + c] * dvx * dvx + D[p.o_w[2] + c] * ax * ax
              + D[p.o_w[3] + c] * dpy * dpy + D[p.o_w[4] + c] * dvy * dvy + D[p.o_w[5] + c] * ay * ay
              + D[p.o_w[6] + c] * ux * ux + D[p.o_w[7] + c] * uy * uy;
      }
    for (int i = 0; i < N; ++i)
      for (int c = 0; c < C; ++c)
        for (int o = 0; o < O; ++o) {
          double v = x[col_so(p, c, o, i)];
          cost += p.w_slack_obs * v * v;
          for (int f = 0; f < 4; ++f) { double w = x[col_sof(p, c, o, i, f)]; cost += p.w_slack_obs * w * w; }
        }
    for (int i = 0; i < N; ++i)
      for (int k1 = 0; k1 < K; ++k1)
        for (int k2 = 0; k2 < K; ++k2)
          for (int q = 0; q < 4; ++q) { double v = x[col_sv(p, k1, k2, i, q)]; cost += p.w_slack * v * v; }
    objective[s] = cost;
  }
}

__global__ void evaluate_kernel(const DevProb *probs, const double *dblob, const int *iblob, int count,
                                const double *xall, double *max_viol /* [count], zeroed */, double *objective /* [count] */) {
  const int s = blockIdx.y;
  if (s >= count) return;
  evaluate_plan(probs, dblob, iblob, s, xall, max_viol, objective);
}

// the plans list[0 .. *n) (streaming runs: the plans harvested in this round; *n is only known on the device)
__global__ void evaluate_list_kernel(const DevProb *probs, const double *dblob, const int *iblob, const int *list, const int *n,
                                     const double *xall, double *max_viol, double *objective) {
  const int nh = *n;
  for (int e = blockIdx.y; e < nh; e += gridDim.y) evaluate_plan(probs, dblob, iblob, list[e], xall, max_viol, objective);
}

// ------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------
void launch_prepare_tables(DevProb *probs, double *dblob, int *iblob, int count, cudaStream_t st) {
  if (count > 0) prepare_tables_kernel<<<count, 128, 0, st>>>(probs, dblob, iblob, count);
}

void launch_assemble_rows(const DevProb *probs, const double *dblob, const int *iblob, int count, long max_rows,
                          long *rowptr, int *cols, double *vals, double *lo, double *hi,
                          unsigned long long *nnz_count, cudaStream_t st) {
  if (count <= 0) return;
  int bx = (int)((max_rows + 255) / 256);
  if (bx < 1) bx = 1;
  if (bx > 148 * 8) bx = 148 * 8;
  dim3 grid(bx, count);
  assemble_rows_kernel<<<grid, 256, 0, st>>>(probs, dblob, iblob, count, rowptr, cols, vals, lo, hi, nnz_count);
}

void launch_evaluate(const DevProb *probs, const double *dblob, const int *iblob, int count, long max_rows,
                     const double *xall, double *max_viol, double *objective, cudaStream_t st) {
  if (count <= 0) return;
  int bx = (int)((max_rows + 255) / 256);
  if (bx < 1) bx = 1;
  if (bx > 64) bx = 64;
  dim3 grid(bx, count);
  evaluate_kernel<<<grid, 256, 0, st>>>(probs, dblob, iblob, count, xall, max_viol, objective);
}

void launch_evaluate_list(const DevProb *probs, const double *dblob, const int *iblob, const int *list, const int *n, int max_n,
                          long max_rows, const double *xall, double *max_viol, double *objective, cudaStream_t st) {
  if (max_n <= 0) return;
  int bx = (int)((max_rows + 255) / 256);
  if (bx < 1) bx = 1;
  if (bx > 64) bx = 64;
  dim3 grid(bx, max_n < HARVEST_GRID / 4 ? max_n : HARVEST_GRID / 4);   // (blocks stride over the plans of the list)
  evaluate_list_kernel<<<grid, 256, 0, st>>>(probs, dblob, iblob, list, n, xall, max_viol, objective);
}

}  // namespace miqp
