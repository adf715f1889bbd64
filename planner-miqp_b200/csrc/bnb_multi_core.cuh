// bnb_multi_core.cuh -- node processing of the multi-car branch and bound (one CTA per node):
// effective regions, node relaxation (node_qp_multi.cuh), scan of the relaxed optimum for the
// least violated alternative of every open disjunction, choice of the branching disjunction.
// Written as barrier-separated phases over work items (see node_qp_multi.cuh), so it also
// compiles for the host with one thread (MQ_EMULATE) for the CPU tests of the logic.
#pragma once
#include "node_qp_multi.cuh"
#include "bnb_common.cuh"

namespace miqp {

// kind: 0 none, 1 mode, 2 env, 3 obs, 4 pair
struct MBranch { int kind, c, i, o, pt, pr, q, ord; double viol; };

MQ_FN void m_offer(MBranch &b, double viol, int ord, int kind, int c, int i, int o, int pt, int pr, int q) {
  if (viol > b.viol || (viol == b.viol && ord < b.ord)) {
    b.viol = viol; b.ord = ord; b.kind = kind; b.c = c; b.i = i; b.o = o; b.pt = pt; b.pr = pr; b.q = q;
  }
}

MQ_FN void m_effective_regions(const MCtx &k) {
  const DevProb &p = *k.p;
  PFOR(c, k.C) {
    int jp = k.I[p.o_initreg + c] - 1;
    k.jeff[c * k.N] = jp;
    for (int i = 1; i < k.N; ++i) {
      const unsigned char m = k.dec[p.off_mode + c * k.N + i];
      const int j = (m == UNDEC) ? -1 : (m == MODE_FROZEN) ? jp : (m >> 2);
      k.jeff[c * k.N + i] = j; jp = j;
    }
  }
  k.sync();
}

MQ_FN double m_mode_alt_violation(const MCtx &k, int c, int i, int alt, int jprev, const double *y) {
  double lo[8], hi[8];
  const int j = (alt == MODE_FROZEN) ? jprev : (alt >> 2);
  m_stage_bounds(k, c, i, j, alt == MODE_FROZEN, lo, hi);
  double v = -MQM_INF;
  for (int t = 1; t < 8; ++t) {
    if (t == Y_PY) continue;
    if (t >= 6 && i == k.N - 1) { if (lo[t] > 0.0) v = fmax(v, lo[t]); if (hi[t] < 0.0) v = fmax(v, -hi[t]); continue; }
    v = fmax(v, y[t] - hi[t]); v = fmax(v, lo[t] - y[t]);
  }
  if (alt != MODE_FROZEN) {
    double a[6], rhs;
    for (int r = 0; r < 5; ++r) {
      m_mode_row(k, alt >> 2, alt & 3, r, a, rhs);
      v = fmax(v, dot6m(a, y) - rhs);
    }
  }
  return v;
}

MQ_FN double m_edge_violation(const double *et, const double *ft, int pt, double sign, const double *y) {
  double a[6], rhs;
  m_edge_row(et, ft, pt, sign, a, rhs);
  return dot6m(a, y) - rhs;
}

// Fills k.imp (a completion of k.dec by the least violated alternatives), k.jeff (effective
// regions of the completion) and the most violated disjunction; returns the number of undecided
// disjunctions.  `bsh` is a shared MBranch used to publish the winner.
MQ_FN int m_scan_node(const MCtx &k, MBranch &br, MBranch *bsh, int ndec_pad) {
  const DevProb &p = *k.p;
  const int C = k.C, N = k.N, O = p.O, E = p.E, L = p.L, nz = k.nz;
  const double tol = 1e-6;
  const int ord_stride = 6 + 5 * O;
  int *bestalt = k.aux, *rdec = k.aux + C * N, *blame = k.aux + 2 * C * N;
  double *bestv = k.auxd;
  PFOR(e, ndec_pad) k.imp[e] = k.dec[e];
  // phase 1: best rho=0 alternative per undecided (car, stage)
  PFOR(it, C * N) {
    const int c = it / N, i = it % N;
    if (i == 0 || k.dec[p.off_mode + c * N + i] != UNDEC) continue;
    const double *y = k.Z + (long)i * nz + 8 * c;
    const int nalt = k.I[p.o_nalt + c];
    const int *alts = k.I + p.o_alt + c * 4 * p.R;
    int best = -1; double bv = MQM_INF;
    for (int a = 0; a < nalt; ++a) {
      const double v = m_mode_alt_violation(k, c, i, alts[a], 0, y);
      if (v < bv - 1e-12) { bv = v; best = alts[a]; }
    }
    bestalt[it] = best; bestv[it] = bv;
  }
  k.sync();
  MBranch mine; mine.kind = 0; mine.viol = tol; mine.ord = 0x7fffffff; mine.c = 0; mine.i = 0; mine.o = 0; mine.pt = 0; mine.pr = 0; mine.q = 0;
  int und = 0;
  // phase 2: region chain of every car (the frozen alternative inherits the region)
  PFOR(c, C) {
    int jp = k.I[p.o_initreg + c] - 1;
    int root_undec = -1;
    k.jeff[c * N] = jp; rdec[c * N] = 1; blame[c * N] = -1;
    for (int i = 1; i < N; ++i) {
      const unsigned char m = k.dec[p.off_mode + c * N + i];
      const double *y = k.Z + (long)i * nz + 8 * c;
      const int ord = (c * N + i) * ord_stride;
      int j;
      if (m == UNDEC || (m == MODE_FROZEN && root_undec >= 0)) {
        const double vfz = m_mode_alt_violation(k, c, i, MODE_FROZEN, jp, y);
        if (m == UNDEC) {
          ++und;
          int best = MODE_FROZEN; double bv = vfz;
          if (bestalt[c * N + i] >= 0 && bestv[c * N + i] < vfz - 1e-12) { best = bestalt[c * N + i]; bv = bestv[c * N + i]; }
          k.imp[p.off_mode + c * N + i] = (unsigned char)best;
          j = (best == MODE_FROZEN) ? jp : (best >> 2);
          root_undec = (best == MODE_FROZEN && root_undec >= 0) ? root_undec : i;
          m_offer(mine, bv, ord, 1, c, i, 0, 0, 0, 0);
        } else {
          j = jp;  // decided frozen, but its region is only implied: blame the chain root
          m_offer(mine, vfz, ord, 1, c, root_undec, 0, 0, 0, 0);
        }
      } else if (m == MODE_FROZEN) {
        j = jp;
      } else { j = m >> 2; root_undec = -1; }
      k.jeff[c * N + i] = j; rdec[c * N + i] = (root_undec < 0); blame[c * N + i] = root_undec;
      jp = j;
    }
  }
  k.sync();
  // phase 3: environment polygons and obstacle edges per point
  PFOR(it, C * N) {
    const int c = it / N, i = it % N;
    if (i == 0) continue;
    const double *y = k.Z + (long)i * nz + 8 * c;
    const int j = k.jeff[it];
    const bool region_decided = rdec[it] != 0;
    const int mode_blame = blame[it];
    const double *ft = k.D + p.o_fronttab + 12 * (c * p.R + j);
    const int ord0 = it * ord_stride;
    if (E > 0)
      for (int pt = 0; pt < 5; ++pt) {
        const unsigned char d = (E == 1) ? (unsigned char)0 : k.dec[p.off_env + it * 5 + pt];
        if (d == UNDEC) ++und;
        if (d != UNDEC && (pt == 0 || region_decided)) continue;
        int best = -1; double bv = MQM_INF;
        for (int e = 0; e < E; ++e) {
          if (d != UNDEC && e != d) continue;
          double v = -MQM_INF;
          for (int ed = k.I[p.o_env_off + e]; ed < k.I[p.o_env_off + e + 1]; ++ed)
            v = fmax(v, m_edge_violation(k.D + p.o_envtab + 3 * ed, ft, pt, -1.0, y));
          if (v < bv) { bv = v; best = e; }
        }
        if (E > 1) k.imp[p.off_env + it * 5 + pt] = (unsigned char)best;
        if (pt > 0 && !region_decided) m_offer(mine, bv, ord0 + 1 + pt, 1, c, mode_blame, 0, 0, 0, 0);
        else m_offer(mine, bv, ord0 + 1 + pt, 2, c, i, 0, pt, 0, 0);
      }
    for (int o = 0; o < O; ++o)
      for (int pt = 0; pt < 5; ++pt) {
        const int off = p.off_obs + ((c * O + o) * N + i) * 5 + pt;
        const unsigned char d = k.dec[off];
        if (d == OBS_SOFT) continue;
        if (d == UNDEC) ++und;
        if (d != UNDEC && (pt == 0 || region_decided)) continue;
        const int ne = k.I[p.o_obs_nedges + o * N + i];
        int best = -1; double bv = MQM_INF;
        for (int ed = 0; ed < ne; ++ed) {
          if (d != UNDEC && ed != d) continue;
          const double v = m_edge_violation(k.D + p.o_obstab + 3 * ((o * N + i) * L + ed), ft, pt, 1.0, y);
          if (v < bv) { bv = v; best = ed; }
        }
        if (ne == 0) { bv = -1.0; best = 0; }
        k.imp[off] = (unsigned char)best;
        if (pt > 0 && !region_decided) m_offer(mine, bv, ord0 + 6 + o * 5 + pt, 1, c, mode_blame, 0, 0, 0, 0);
        else m_offer(mine, bv, ord0 + 6 + o * 5 + pt, 3, c, i, o, pt, 0, 0);
      }
  }
  // phase 4: collision sides of every pair quadruple (stage 0 is never branched on: the state is
  // fixed there; its sides are taken by the completion)
  if (k.P > 0) {
    const int ordp = C * N * ord_stride;
    PFOR(i, N) {
      int pr = 0;
      for (int a = 0; a < C - 1; ++a)
        for (int b = a + 1; b < C; ++b, ++pr) {
          const int ja = k.jeff[a * N + i], jb = k.jeff[b * N + i];
          const bool rda = (i == 0) || rdec[a * N + i] != 0, rdb = (i == 0) || rdec[b * N + i] != 0;
          const double *ya = k.Z + (long)i * nz + 8 * a, *yb = k.Z + (long)i * nz + 8 * b;
          for (int q = 0; q < 4; ++q) {
            const int off = p.off_pair + (pr * N + i) * 4 + q;
            const unsigned char d = k.dec[off];
            if (d == UNDEC) ++und;
            const bool need_a = (q == 2 || q == 3), need_b = (q == 1 || q == 3);
            const bool enforced = (d != UNDEC) && (!need_a || rda) && (!need_b || rdb);
            if (enforced) continue;
            // slack of this quadruple (if it carries one and its row is not in the relaxation) is 0
            int best = -1; double bv = MQM_INF;
            for (int side = 0; side < 4; ++side) {
              if (d != UNDEC && side != d) continue;
              PairRow r; m_pair_row(k, a, b, i, q, side, ja, jb, r);
              const double v = dot6m(r.ca, ya) + dot6m(r.cb, yb) - r.rhs;
              if (v < bv) { bv = v; best = side; }
            }
            k.imp[off] = (unsigned char)best;
            if (i == 0) continue;
            const int ord = ordp + (pr * N + i) * 4 + q;
            if (need_a && !rda) m_offer(mine, bv, ord, 1, a, blame[a * N + i], 0, 0, 0, 0);
            else if (need_b && !rdb) m_offer(mine, bv, ord, 1, b, blame[b * N + i], 0, 0, 0, 0);
            else m_offer(mine, bv, ord, 4, 0, i, 0, 0, pr, q);
          }
        }
    }
  }
  // phase 5: most violated, first in scan order among equals
  const double vbest = k.rmax(mine.viol);
  const double obest = -k.rmax((mine.viol == vbest) ? -(double)mine.ord : -4e9);
  if (mine.viol == vbest && (double)mine.ord == obest) *bsh = mine;
  und = k.rsumi(und);   // (barriers: *bsh is visible afterwards)
  br = *bsh;
  k.sync();
  return und;
}

// ---------------------------------------------------------------------------------------
// lower bound of a child before it is solved: the parent's optimum z* violates row g.z <= h of the
// child's alternative by v > 0; every point of the child then costs at least
//     f(z*) + 1/2 v^2 / (g' W_i g)          (W_i: reach table of formulation_tables.cuh)
// because f(z) >= f(z*) + 1/2 d'Qd for every z = z* + d of the parent's feasible set (z* optimal,
// f quadratic) and d has to move by v against g at step i.  The largest such term over the rows of
// the alternative is added to the parent's objective; children whose bound reaches the cutoff are
// never created.
// ---------------------------------------------------------------------------------------
MQ_FN double m_quad_w(const MCtx &k, int c, int i, const double a[6]) {
  const double *t = k.D + k.p->o_wtab + 14 * (c * k.N + i);
  double g = 0.0;
  for (int ax = 0; ax < 2; ++ax) {
    const double *w = t + 7 * ax; const double *v = a + 3 * ax;
    g += w[0] * v[0] * v[0] + 2.0 * w[1] * v[1] * v[0] + w[2] * v[1] * v[1] + 2.0 * w[3] * v[2] * v[0] + 2.0 * w[4] * v[2] * v[1] + w[5] * v[2] * v[2];
  }
  return g;
}
MQ_FN double m_delta(double viol, double G) {
  if (!(viol > 1e-7) || !(G > 1e-14)) return 0.0;
  return 0.5 * viol * viol / G;
}
MQ_FN double m_bound_delta(const MCtx &k, int c, int i, int T, double viol) {
  const double *t = k.D + k.p->o_wtab + 14 * (c * k.N + i);
  double G;
  if (T < 6) { const int o = T % 3; G = t[7 * (T / 3) + (o == 0 ? 0 : o == 1 ? 2 : 5)]; }
  else G = t[7 * (T - 6) + 6];
  return m_delta(viol, G);
}

// increase of the lower bound for alternative `alt` of the branching disjunction br (>= 0)
MQ_FN double m_alt_delta(const MCtx &k, const MBranch &br, int alt) {
  const DevProb &p = *k.p;
  const int N = k.N, C = k.C;
  const int *rdec = k.aux + C * N;
  double dl = 0.0;
  if (br.kind == 1) {
    const int c = br.c, i = br.i;
    const double *y = k.Z + (long)i * k.nz + 8 * c;
    const bool frozen = (alt == MODE_FROZEN);
    const int j = frozen ? (rdec[c * N + i - 1] ? k.jeff[c * N + i - 1] : -1) : (alt >> 2);
    double lo[8], hi[8];
    m_stage_bounds(k, c, i, j, frozen, lo, hi);
    for (int t = 1; t < 8; ++t) {
      if (t == Y_PY) continue;
      if (t >= 6 && i == N - 1) continue;
      dl = fmax(dl, m_bound_delta(k, c, i, t, y[t] - hi[t]));
      dl = fmax(dl, m_bound_delta(k, c, i, t, lo[t] - y[t]));
    }
    if (!frozen) {
      double a[6], rhs;
      for (int r = 0; r < 5; ++r) { m_mode_row(k, alt >> 2, alt & 3, r, a, rhs); dl = fmax(dl, m_delta(dot6m(a, y) - rhs, m_quad_w(k, c, i, a))); }
    }
  } else if (br.kind == 2) {
    const int c = br.c, i = br.i;
    const double *y = k.Z + (long)i * k.nz + 8 * c;
    const double *ft = k.D + p.o_fronttab + 12 * (c * p.R + (k.jeff[c * N + i] >= 0 ? k.jeff[c * N + i] : 0));
    double a[6], rhs;
    for (int ed = k.I[p.o_env_off + alt]; ed < k.I[p.o_env_off + alt + 1]; ++ed) {
      m_edge_row(k.D + p.o_envtab + 3 * ed, ft, br.pt, -1.0, a, rhs);
      dl = fmax(dl, m_delta(dot6m(a, y) - rhs, m_quad_w(k, c, i, a)));
    }
  } else if (br.kind == 3) {
    if (alt == OBS_SOFT) return p.w_slack_obs;
    const int c = br.c, i = br.i;
    const double *y = k.Z + (long)i * k.nz + 8 * c;
    const double *ft = k.D + p.o_fronttab + 12 * (c * p.R + (k.jeff[c * N + i] >= 0 ? k.jeff[c * N + i] : 0));
    double a[6], rhs;
    m_edge_row(k.D + p.o_obstab + 3 * ((br.o * N + i) * p.L + alt), ft, br.pt, 1.0, a, rhs);
    dl = m_delta(dot6m(a, y) - rhs, m_quad_w(k, c, i, a));
  } else if (br.kind == 4) {
    int a = 0, rem = br.pr;
    while (rem >= C - 1 - a) { rem -= C - 1 - a; ++a; }
    const int b = a + 1 + rem, i = br.i;
    PairRow r; m_pair_row(k, a, b, i, br.q, alt, k.jeff[a * N + i], k.jeff[b * N + i], r);
    const double *ya = k.Z + (long)i * k.nz + 8 * a, *yb = k.Z + (long)i * k.nz + 8 * b;
    double G = m_quad_w(k, a, i, r.ca) + m_quad_w(k, b, i, r.cb);
    if (r.slack >= 0 && m_slack_cap(k, i) > 1e-12 && p.w_slack > 0.0) G += 1.0 / (2.0 * p.w_slack);
    dl = m_delta(dot6m(r.ca, ya) + dot6m(r.cb, yb) - r.rhs, G);
  }
  return dl;
}

// outcome of one node
enum { MN_INFEASIBLE = 0, MN_PRUNED, MN_INCUMBENT, MN_BRANCH, MN_UNKNOWN };
// obj: valid lower bound of the node; fval: objective of the point in Z (an upper bound of the relaxation, = obj if converged);
// est: ordering hint of the children (the dive follows it; bounds and pruning never use it)
struct MNodeOut { int what, iters, nalt, soff, converged; long rows; double obj, fval, pruned_min; bool from_imp; };

// Shared scratch of the node processing that is not part of the QP workspace
struct MShared { MBranch br; int nkeep; double pruned_min; unsigned char alts[260]; double cb[260]; };

// k.dec holds the node; returns what to do with it.  For MN_BRANCH the children are
// copies of (from_imp ? k.imp : k.dec) with byte soff (if >= 0) set to sh->alts[0..nalt).
MQ_FN MNodeOut m_process_node(const MCtx &k, MShared *sh, double nbound, double cutoff, int ndec_pad) {
  const DevProb &p = *k.p;
  MNodeOut out; out.what = MN_INFEASIBLE; out.iters = 0; out.nalt = 0; out.soff = -1; out.rows = 0; out.obj = 0.0; out.from_imp = false;
  out.pruned_min = MQM_INF;
  m_effective_regions(k);
  int nsoft = 0;
  PFOR(e, 5 * k.C * p.O * k.N) nsoft += (k.dec[p.off_obs + e] == OBS_SOFT);
  nsoft = k.rsumi(nsoft);
  const double pen = nsoft * p.w_slack_obs;
  const MQpResult r = m_solve_node_qp(k);
  out.iters = r.iters; out.rows = r.rows; out.converged = r.converged;
  if (r.status == 1) return out;                               // proven infeasible
  if (r.status != 0) { out.what = MN_UNKNOWN; out.obj = nbound; return out; }   // neither solved nor refuted
  // a stalled relaxation is only a feasible point: its objective is an upper bound of the relaxation; the node's lower
  // bound is the Lagrangian bound of the multipliers (or the parent's bound)
  const double fval = r.obj + pen;
  double obj = r.converged ? fval : fmax(nbound, r.lb + pen);
  if (obj < nbound) obj = nbound;  // numerical monotonicity
  out.obj = obj; out.fval = fval > obj ? fval : obj;
  if (obj >= cutoff) { out.what = MN_PRUNED; return out; }
  MBranch br;
  const int und = m_scan_node(k, br, &sh->br, ndec_pad);
  // (a stalled point that satisfies an alternative of every disjunction is still replaced by its completion alone; the
  // dropped completions are accounted for by the caller: pruned_min = obj)
  if (br.kind == 0 && und > 0 && !r.converged) out.pruned_min = obj;
  if (br.kind == 0 && und == 0) { out.what = MN_INCUMBENT; return out; }
  out.what = MN_BRANCH;
  if (br.kind == 0) { out.nalt = 1; out.from_imp = true; out.soff = -1; if (k.tid == 0) sh->cb[0] = obj; k.sync(); return out; }
  out.nalt = branch_alts(p, k.I, br.kind, br.c, br.i, br.o, br.pt, br.pr, br.q, out.soff, k.tid == 0 ? sh->alts : nullptr);
  k.sync();
  // child bounds; children that reach the cutoff are dropped here
  PFOR(a, out.nalt) sh->cb[a] = r.converged ? fmax(obj, fval + 0.999 * m_alt_delta(k, br, sh->alts[a])) : obj;
  k.sync();
  if (k.tid == 0) sh->nkeep = drop_cut_children(sh->alts, sh->cb, out.nalt, cutoff, sh->pruned_min);
  k.sync();
  out.nalt = sh->nkeep; out.pruned_min = sh->pruned_min;
  k.sync();
  return out;
}

}  // namespace miqp
