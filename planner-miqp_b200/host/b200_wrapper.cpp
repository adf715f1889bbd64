// b200_wrapper.cpp -- see b200_wrapper.hpp.  Host driver of libmiqp_b200.so in the shape of the
// reference's CplexWrapper (src/cplex_wrapper.cpp).
#include "b200_wrapper.hpp"
#include "dat_reader.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <fstream>
#include <iomanip>
#include <limits>
#include <sstream>
#include <cstdlib>
#include <initializer_list>

namespace miqp {
namespace planner {
namespace cplex {

namespace {

// RoundWithPrecision of the reference (src/model_input_data_source.hpp:74-79)
inline double RoundDecimals(double v, int decimals) {
  if (decimals <= 0) return v;
  const double scale = std::pow(10.0, decimals);
  return std::round(v * scale) / scale;
}

struct Flattener {
  FlatProblem &f;
  int dec;
  const double *vec(const VectorXd &v) { return raw(v.data(), v.size()); }
  const double *mat(const MatrixXd &m) { return raw(m.data(), m.size()); }
  const double *raw(const double *src, int n) {
    f.d.emplace_back(std::max(n, 1), 0.0);
    for (int k = 0; k < n; ++k) f.d.back()[k] = RoundDecimals(src[k], dec);
    return f.d.back().data();
  }
  const int *ints(const int *src, int n) {
    f.i.emplace_back(std::max(n, 1), 0);
    for (int k = 0; k < n; ++k) f.i.back()[k] = src[k];
    return f.i.back().data();
  }
  double num(float v) { return RoundDecimals((double)v, dec); }
};

// closed edge list of a (k, 2) vertex matrix: edge e runs from vertex e to vertex e+1, the last one
// closes the polygon (addLineSet, src/model_input_data_source.cpp:167-178)
void AppendEdges(const MatrixXd &v, int dec, std::vector<double> &out, int pad_to) {
  const int k = v.rows();
  for (int e = 0; e < k; ++e) {
    const int n = (e + 1) % k;
    out.push_back(RoundDecimals(v(e, 0), dec)); out.push_back(RoundDecimals(v(e, 1), dec));
    out.push_back(RoundDecimals(v(n, 0), dec)); out.push_back(RoundDecimals(v(n, 1), dec));
  }
  for (int e = k; e < pad_to; ++e) for (int t = 0; t < 4; ++t) out.push_back(0.0);
}

}  // namespace

void Flatten(const ModelParameters &m, int precision, FlatProblem &out) {
  out.d.clear(); out.i.clear();
  out.d.reserve(64); out.i.reserve(8);   // pointers into the inner vectors stay valid either way
  Flattener F{out, precision > 2 ? precision - 2 : 0};
  MiqpB200Problem &p = out.p;
  p = MiqpB200Problem{};
  p.N = m.NumSteps; p.R = m.nr_regions; p.C = m.NumCars;
  p.O = m.nr_obstacles; p.L = m.nr_obstacles > 0 ? m.max_lines_obstacles : 0; p.E = m.nr_environments;
  p.ts = F.num(m.ts);
  p.min_vel = F.num(m.min_vel_x_y); p.max_vel = F.num(m.max_vel_x_y);
  p.total_min_acc = F.num(m.total_min_acc); p.total_max_acc = F.num(m.total_max_acc);
  p.total_min_jerk = F.num(m.total_min_jerk); p.total_max_jerk = F.num(m.total_max_jerk);
  p.maximum_slack = F.num(m.maximum_slack);
  p.w_slack = F.num(m.WEIGHTS_SLACK); p.w_slack_obs = F.num(m.WEIGHTS_SLACK_OBSTACLE);
  p.min_region_change_speed = F.num(m.minimum_region_change_speed);
  p.gap_tol = F.num(m.relative_mip_gap_tolerance); p.time_limit = F.num(m.max_solution_time);
  p.safety = F.vec(m.agent_safety_distance); p.safety_slack = F.vec(m.agent_safety_distance_slack);
  p.w_pos_x = F.vec(m.WEIGHTS_POS_X); p.w_vel_x = F.vec(m.WEIGHTS_VEL_X); p.w_acc_x = F.vec(m.WEIGHTS_ACC_X);
  p.w_pos_y = F.vec(m.WEIGHTS_POS_Y); p.w_vel_y = F.vec(m.WEIGHTS_VEL_Y); p.w_acc_y = F.vec(m.WEIGHTS_ACC_Y);
  p.w_jerk_x = F.vec(m.WEIGHTS_JERK_X); p.w_jerk_y = F.vec(m.WEIGHTS_JERK_Y);
  p.wheelbase = F.vec(m.WheelBase); p.radius = F.vec(m.CollisionRadius);
  p.x0 = F.mat(m.IntitialState);
  p.x_ref = F.mat(m.x_ref); p.vx_ref = F.mat(m.vx_ref); p.y_ref = F.mat(m.y_ref); p.vy_ref = F.mat(m.vy_ref);
  p.min_acc_x = F.mat(m.acc_limit_params.min_x); p.max_acc_x = F.mat(m.acc_limit_params.max_x);
  p.min_acc_y = F.mat(m.acc_limit_params.min_y); p.max_acc_y = F.mat(m.acc_limit_params.max_y);
  p.min_jerk_x = F.mat(m.jerk_limit_params.min_x); p.max_jerk_x = F.mat(m.jerk_limit_params.max_x);
  p.min_jerk_y = F.mat(m.jerk_limit_params.min_y); p.max_jerk_y = F.mat(m.jerk_limit_params.max_y);
  p.initial_region = F.ints(m.initial_region.data(), m.initial_region.size());
  p.possible_region = F.ints(m.possible_region.data(), m.possible_region.size());
  // obstacles: [O][N][L][4] edges; an obstacle that carries fewer than N polygons repeats its last one
  {
    std::vector<double> edges; std::vector<int> nedges;
    for (int o = 0; o < p.O; ++o) {
      const std::vector<MatrixXd> &poly = m.ObstacleConvexPolygon[o];
      for (int i = 0; i < p.N; ++i) {
        if (poly.empty()) { nedges.push_back(0); AppendEdges(MatrixXd(), F.dec, edges, p.L); continue; }
        const MatrixXd &v = poly[std::min<size_t>(i, poly.size() - 1)];
        if (v.rows() > p.L) throw std::invalid_argument("obstacle polygon has more edges than max_lines_obstacles");
        nedges.push_back(v.rows());
        AppendEdges(v, F.dec, edges, p.L);
      }
    }
    out.d.push_back(edges.empty() ? std::vector<double>(4, 0.0) : edges); p.obs_edges = out.d.back().data();
    p.obs_nedges = F.ints(nedges.data(), (int)nedges.size());
    p.obs_soft = F.ints(m.obstacle_is_soft.data(), (int)m.obstacle_is_soft.size());
  }
  {
    std::vector<double> edges; std::vector<int> off{0};
    for (int e = 0; e < p.E; ++e) {
      AppendEdges(m.MultiEnvironmentConvexPolygon[e], F.dec, edges, 0);
      off.push_back((int)edges.size() / 4);
    }
    out.d.push_back(edges.empty() ? std::vector<double>(4, 0.0) : edges); p.env_edges = out.d.back().data();
    p.env_off = F.ints(off.data(), (int)off.size());
  }
  p.frac = F.mat(m.fraction_parameters);
  p.poly_sint_ub = F.mat(m.poly_orientation_params.POLY_SINT_UB); p.poly_sint_lb = F.mat(m.poly_orientation_params.POLY_SINT_LB);
  p.poly_coss_ub = F.mat(m.poly_orientation_params.POLY_COSS_UB); p.poly_coss_lb = F.mat(m.poly_orientation_params.POLY_COSS_LB);
  p.poly_kappa_max = F.mat(m.poly_curvature_params.POLY_KAPPA_AX_MAX); p.poly_kappa_min = F.mat(m.poly_curvature_params.POLY_KAPPA_AX_MIN);
}

// ---------------------------------------------------------------------------------------
namespace {
template <class F> void ForEachFamily(const MiqpB200Layout &l, RawResults &r, F &&f) {
  const int C = l.C, N = l.N, R = l.R, O = l.O, L = l.L, E = l.E, K = l.K;
  Tensor<double, 2> *core[12] = {&r.u_x, &r.u_y, &r.pos_x, &r.vel_x, &r.acc_x, &r.pos_y, &r.vel_y, &r.acc_y,
                                 &r.pos_x_front_UB, &r.pos_x_front_LB, &r.pos_y_front_UB, &r.pos_y_front_LB};
  for (int b = 0; b < 12; ++b) { core[b]->resize(C, N); f(core[b]->data(), (long)b * C * N, (long)C * N, 1, -1, false); }
  Tensor<int, 3> *nwe[5] = {&r.notWithinEnvironmentRear, &r.notWithinEnvironmentFrontUbUb, &r.notWithinEnvironmentFrontLbUb,
                            &r.notWithinEnvironmentFrontUbLb, &r.notWithinEnvironmentFrontLbLb};
  for (int k = 0; k < 5; ++k) { nwe[k]->resize(C, E, N); f(nwe[k]->data(), l.base_nwe + (long)k * C * E * N, (long)C * E * N, 1, N, true); }
  r.active_region.resize(C, N, R); f(r.active_region.data(), l.base_ar, (long)C * N * R, R, N, true);
  Tensor<int, 2> *rc[5] = {&r.region_change_not_allowed_x_positive, &r.region_change_not_allowed_y_positive,
                           &r.region_change_not_allowed_x_negative, &r.region_change_not_allowed_y_negative,
                           &r.region_change_not_allowed_combined};
  for (int k = 0; k < 5; ++k) { rc[k]->resize(C, N); f(rc[k]->data(), l.base_rcna + (long)k * C * N, (long)C * N, 1, N, true); }
  r.deltacc.resize(C, O, N, L); f(r.deltacc.data(), l.base_dcc, (long)C * O * N * L, L, N, true);
  r.deltacc_front.resize(C, O, N, L, 4); f(r.deltacc_front.data(), l.base_dcf, (long)C * O * N * L * 4, L * 4, N, true);
  r.slackvarsObstacle.resize(C, O, N); f(r.slackvarsObstacle.data(), l.base_so, (long)C * O * N, 1, N, false);
  r.slackvarsObstacle_front.resize(C, O, N, 4); f(r.slackvarsObstacle_front.data(), l.base_sof, (long)C * O * N * 4, 4, N, false);
  r.car2car_collision.resize(K, K, N, 16); f(r.car2car_collision.data(), l.base_c2c, (long)K * K * N * 16, 16, N, true);
  r.slackvars.resize(K, K, N, 4); f(r.slackvars.data(), l.base_sv, (long)K * K * N * 4, 4, N, false);
  r.N = N; r.NrEnvironments = E; r.NrRegions = R; r.NrObstacles = O; r.MaxLinesObstacles = L;
  r.NrCarToCarCollisions = K; r.NrCars = C;
}
}  // namespace

void Unpack(const MiqpB200Layout &l, const double *x, RawResults &r) {
  struct {
    const double *x;
    void operator()(double *dst, long base, long n, int, int, bool) { for (long k = 0; k < n; ++k) dst[k] = x[base + k]; }
    // binaries are rounded; the slack families are truncated like the reference's double -> int copy
    void operator()(int *dst, long base, long n, int, int, bool binary) {
      for (long k = 0; k < n; ++k) dst[k] = binary ? (int)std::lround(x[base + k]) : (int)x[base + k];
    }
  } f{x};
  ForEachFamily(l, r, f);
}

void Pack(const MiqpB200Layout &l, const RawResults &rr, bool relax_last_step, std::vector<double> &x) {
  x.assign(l.ncols, 0.0);
  // families in layout order, read from rr directly
  const int C = l.C, N = l.N, R = l.R, O = l.O, L = l.L, E = l.E, K = l.K;
  auto put_d = [&](const Tensor<double, 2> &t, long base) {
    if ((long)t.size() != (long)C * N) return;
    for (long k = 0; k < (long)C * N; ++k) x[base + k] = t.data()[k];
  };
  const Tensor<double, 2> *core[12] = {&rr.u_x, &rr.u_y, &rr.pos_x, &rr.vel_x, &rr.acc_x, &rr.pos_y, &rr.vel_y, &rr.acc_y,
                                       &rr.pos_x_front_UB, &rr.pos_x_front_LB, &rr.pos_y_front_UB, &rr.pos_y_front_LB};
  for (int b = 0; b < 12; ++b) put_d(*core[b], (long)b * C * N);
  const double nan = std::numeric_limits<double>::quiet_NaN();
  // inner = entries per time step behind the step index; a family whose tensor has the wrong size stays undecided
  auto put_i = [&](const int *src, size_t have, long base, long n, int inner, bool binary) {
    if ((long)have != n) { if (binary) for (long k = 0; k < n; ++k) x[base + k] = nan; return; }
    for (long k = 0; k < n; ++k) {
      const bool last = ((k / inner) % N) == N - 1;
      x[base + k] = (binary && relax_last_step && last) ? nan : (double)src[k];
    }
  };
  const Tensor<int, 3> *nwe[5] = {&rr.notWithinEnvironmentRear, &rr.notWithinEnvironmentFrontUbUb, &rr.notWithinEnvironmentFrontLbUb,
                                  &rr.notWithinEnvironmentFrontUbLb, &rr.notWithinEnvironmentFrontLbLb};
  for (int k = 0; k < 5; ++k) put_i(nwe[k]->data(), nwe[k]->size(), l.base_nwe + (long)k * C * E * N, (long)C * E * N, 1, true);
  put_i(rr.active_region.data(), rr.active_region.size(), l.base_ar, (long)C * N * R, R, true);
  const Tensor<int, 2> *rc[5] = {&rr.region_change_not_allowed_x_positive, &rr.region_change_not_allowed_y_positive,
                                 &rr.region_change_not_allowed_x_negative, &rr.region_change_not_allowed_y_negative,
                                 &rr.region_change_not_allowed_combined};
  for (int k = 0; k < 5; ++k) put_i(rc[k]->data(), rc[k]->size(), l.base_rcna + (long)k * C * N, (long)C * N, 1, true);
  put_i(rr.deltacc.data(), rr.deltacc.size(), l.base_dcc, (long)C * O * N * L, std::max(L, 1), true);
  put_i(rr.deltacc_front.data(), rr.deltacc_front.size(), l.base_dcf, (long)C * O * N * L * 4, std::max(L * 4, 1), true);
  put_i(rr.slackvarsObstacle.data(), rr.slackvarsObstacle.size(), l.base_so, (long)C * O * N, 1, false);
  put_i(rr.slackvarsObstacle_front.data(), rr.slackvarsObstacle_front.size(), l.base_sof, (long)C * O * N * 4, 4, false);
  put_i(rr.car2car_collision.data(), rr.car2car_collision.size(), l.base_c2c, (long)K * K * N * 16, 16, true);
  put_i(rr.slackvars.data(), rr.slackvars.size(), l.base_sv, (long)K * K * N * 4, 4, false);
}

// ---------------------------------------------------------------------------------------
bool WriteParametersDat(const MiqpB200Problem &p, const ModelParameters &m, const std::string &path) {
  std::ofstream f(path);
  if (!f.good()) return false;
  f << std::setprecision(12);   // the reference prints its dumps with 12 display digits (src/cplex_wrapper.hpp:109-110)
  auto vec = [&](const char *name, const double *a, int n) {
    f << name << " = [";
    for (int k = 0; k < n; ++k) f << (k ? " " : "") << a[k];
    f << "];\n";
  };
  auto mat = [&](const char *name, const double *a, int r, int c) {
    f << name << " = [";
    for (int i = 0; i < r; ++i) { f << (i ? "\n" : "") << "["; for (int j = 0; j < c; ++j) f << (j ? " " : "") << a[(long)i * c + j]; f << "]"; }
    f << "];\n";
  };
  auto edgeset = [&](const double *e, int n) {
    f << "{";
    for (int k = 0; k < n; ++k) f << (k ? "\n" : "") << "<" << (k + 1) << " " << e[4 * k] << " " << e[4 * k + 1] << " " << e[4 * k + 2] << " " << e[4 * k + 3] << ">";
    f << "}";
  };
  f << "NumSteps = " << p.N << ";\nnr_environments = " << p.E << ";\nnr_regions = " << p.R << ";\nnr_obstacles = " << p.O
    << ";\nmax_lines_obstacles = " << p.L << ";\nNumCars = " << p.C << ";\n";
  f << "max_solution_time = " << p.time_limit << ";\nrelative_mip_gap_tolerance = " << p.gap_tol << ";\n";
  f << "mipdisplay = " << m.mipdisplay << ";\nmipemphasis = " << m.mipemphasis << ";\nrelobjdif = " << (double)m.relobjdif << ";\n";
  f << "cutpass = " << m.cutpass << ";\nprobe = " << m.probe << ";\nrepairtries = " << m.repairtries << ";\nrinsheur = " << m.rinsheur
    << ";\nvarsel = " << m.varsel << ";\nmircuts = " << m.mircuts << ";\nparallelmode = " << m.parallelmode << ";\n";
  f << "ts = " << p.ts << ";\nmin_vel_x_y = " << p.min_vel << ";\nmax_vel_x_y = " << p.max_vel << ";\ntotal_min_acc = " << p.total_min_acc
    << ";\ntotal_max_acc = " << p.total_max_acc << ";\ntotal_min_jerk = " << p.total_min_jerk << ";\ntotal_max_jerk = " << p.total_max_jerk << ";\n";
  vec("agent_safety_distance", p.safety, p.N); vec("agent_safety_distance_slack", p.safety_slack, p.N);
  f << "maximum_slack = " << p.maximum_slack << ";\n";
  vec("WEIGHTS_POS_X", p.w_pos_x, p.C); vec("WEIGHTS_VEL_X", p.w_vel_x, p.C); vec("WEIGHTS_ACC_X", p.w_acc_x, p.C);
  vec("WEIGHTS_POS_Y", p.w_pos_y, p.C); vec("WEIGHTS_VEL_Y", p.w_vel_y, p.C); vec("WEIGHTS_ACC_Y", p.w_acc_y, p.C);
  vec("WEIGHTS_JERK_X", p.w_jerk_x, p.C); vec("WEIGHTS_JERK_Y", p.w_jerk_y, p.C);
  f << "WEIGHTS_SLACK = " << p.w_slack << ";\nWEIGHTS_SLACK_OBSTACLE = " << p.w_slack_obs << ";\n";
  vec("WheelBase", p.wheelbase, p.C); vec("CollisionRadius", p.radius, p.C);
  mat("IntitialState", p.x0, p.C, 6);
  mat("x_ref", p.x_ref, p.C, p.N); mat("vx_ref", p.vx_ref, p.C, p.N); mat("y_ref", p.y_ref, p.C, p.N); mat("vy_ref", p.vy_ref, p.C, p.N);
  mat("min_acc_x", p.min_acc_x, p.C, p.R); mat("max_acc_x", p.max_acc_x, p.C, p.R);
  mat("min_acc_y", p.min_acc_y, p.C, p.R); mat("max_acc_y", p.max_acc_y, p.C, p.R);
  mat("min_jerk_x", p.min_jerk_x, p.C, p.R); mat("max_jerk_x", p.max_jerk_x, p.C, p.R);
  mat("min_jerk_y", p.min_jerk_y, p.C, p.R); mat("max_jerk_y", p.max_jerk_y, p.C, p.R);
  f << "initial_region = [";
  for (int c = 0; c < p.C; ++c) f << (c ? " " : "") << p.initial_region[c];
  f << "];\npossible_region = [";
  for (int c = 0; c < p.C; ++c) { f << (c ? "\n" : "") << "["; for (int j = 0; j < p.R; ++j) f << (j ? " " : "") << p.possible_region[c * p.R + j]; f << "]"; }
  f << "];\nObstacleConvexPolygon = [";
  for (int o = 0; o < p.O; ++o) {
    f << (o ? "\n" : "") << "[";
    for (int i = 0; i < p.N; ++i) { f << (i ? " " : ""); edgeset(p.obs_edges + ((long)(o * p.N + i) * p.L) * 4, p.obs_nedges[o * p.N + i]); }
    f << "]";
  }
  f << "];\nobstacle_is_soft = [";
  for (int o = 0; o < p.O; ++o) f << (o ? " " : "") << p.obs_soft[o];
  f << "];\nMultiEnvironmentConvexPolygon = [";
  for (int e = 0; e < p.E; ++e) { f << (e ? " " : ""); edgeset(p.env_edges + 4L * p.env_off[e], p.env_off[e + 1] - p.env_off[e]); }
  f << "];\n";
  mat("fraction_parameters", p.frac, p.R, 4);
  f << "minimum_region_change_speed = " << p.min_region_change_speed << ";\n";
  mat("POLY_SINT_UB", p.poly_sint_ub, p.R, 3); mat("POLY_SINT_LB", p.poly_sint_lb, p.R, 3);
  mat("POLY_COSS_UB", p.poly_coss_ub, p.R, 3); mat("POLY_COSS_LB", p.poly_coss_lb, p.R, 3);
  mat("POLY_KAPPA_AX_MAX", p.poly_kappa_max, p.R, 3); mat("POLY_KAPPA_AX_MIN", p.poly_kappa_min, p.R, 3);
  return f.good();
}

// ---------------------------------------------------------------------------------------
B200Wrapper::B200Wrapper() : B200Wrapper(12) {}
B200Wrapper::B200Wrapper(int precision) : results_(std::make_shared<RawResults>()), precision_(precision) {}
B200Wrapper::B200Wrapper(const std::string &modpath, const std::string &, ParameterSource source, int precision) : B200Wrapper(precision) {
  source_ = source; modPath_ = modpath;
}
B200Wrapper::B200Wrapper(const B200Wrapper &o)
    : parameters_(o.parameters_), results_(std::make_shared<RawResults>()), precision_(o.precision_), device_(o.device_),
      useSos_(o.useSos_), useBranchingPriorities_(o.useBranchingPriorities_), bufferOutputs_(o.bufferOutputs_),
      debugPrint_(o.debugPrint_), collectSizes_(o.collectSizes_), prioStart_(o.prioStart_), prioExtent_(o.prioExtent_),
      debugPath_(o.debugPath_), debugPrefix_(o.debugPrefix_), source_(o.source_), modPath_(o.modPath_), datFile_(o.datFile_),
      poolCapacity_(o.poolCapacity_) {}
B200Wrapper &B200Wrapper::operator=(const B200Wrapper &o) { debugPath_ = o.debugPath_; return *this; }
B200Wrapper::~B200Wrapper() { if (solver_) miqp_b200_destroy(solver_); }

void B200Wrapper::overrideSolverSettingsDataSource(std::shared_ptr<ModelParameters> o) {
  if (!o) return;
  if (!parameters_) parameters_ = std::make_shared<ModelParameters>();
  parameters_->max_solution_time = o->max_solution_time;
  parameters_->relative_mip_gap_tolerance = o->relative_mip_gap_tolerance;
  parameters_->mipdisplay = o->mipdisplay; parameters_->mipemphasis = o->mipemphasis;
  parameters_->relobjdif = o->relobjdif; parameters_->cutpass = o->cutpass; parameters_->probe = o->probe;
  parameters_->repairtries = o->repairtries; parameters_->rinsheur = o->rinsheur; parameters_->varsel = o->varsel;
  parameters_->mircuts = o->mircuts; parameters_->parallelmode = o->parallelmode;
}

// ---- column names, .mst, .lp -------------------------------------------------------------------------------------------
std::vector<std::string> ColumnNames(const MiqpB200Layout &l) {
  std::vector<std::string> n((size_t)l.ncols);
  auto idx = [](std::initializer_list<int> v) { std::string s; for (int k : v) s += "(" + std::to_string(k + 1) + ")"; return s; };
  static const char *core[12] = {"u_x", "u_y", "pos_x", "vel_x", "acc_x", "pos_y", "vel_y", "acc_y",
                                 "pos_x_front_UB", "pos_x_front_LB", "pos_y_front_UB", "pos_y_front_LB"};
  static const char *nwe[5] = {"notWithinEnvironmentRear", "notWithinEnvironmentFrontUbUb", "notWithinEnvironmentFrontLbUb",
                               "notWithinEnvironmentFrontUbLb", "notWithinEnvironmentFrontLbLb"};
  static const char *rcna[5] = {"region_change_not_allowed_x_positive", "region_change_not_allowed_y_positive",
                                "region_change_not_allowed_x_negative", "region_change_not_allowed_y_negative",
                                "region_change_not_allowed_combined"};
  const int C = l.C, N = l.N, R = l.R, O = l.O, L = l.L, E = l.E, K = l.K;
  for (int b = 0; b < 12; ++b) for (int c = 0; c < C; ++c) for (int i = 0; i < N; ++i) n[((size_t)b * C + c) * N + i] = core[b] + idx({c, i});
  for (int k = 0; k < 5; ++k) for (int c = 0; c < C; ++c) for (int e = 0; e < E; ++e) for (int i = 0; i < N; ++i)
    n[l.base_nwe + (((size_t)k * C + c) * E + e) * N + i] = nwe[k] + idx({c, e, i});
  for (int c = 0; c < C; ++c) for (int i = 0; i < N; ++i) for (int j = 0; j < R; ++j) n[l.base_ar + ((size_t)c * N + i) * R + j] = "active_region" + idx({c, i, j});
  for (int k = 0; k < 5; ++k) for (int c = 0; c < C; ++c) for (int i = 0; i < N; ++i) n[l.base_rcna + ((size_t)k * C + c) * N + i] = rcna[k] + idx({c, i});
  for (int c = 0; c < C; ++c) for (int o = 0; o < O; ++o) for (int i = 0; i < N; ++i) {
    for (int e = 0; e < L; ++e) {
      n[l.base_dcc + (((size_t)c * O + o) * N + i) * L + e] = "deltacc" + idx({c, o, i, e});
      for (int f = 0; f < 4; ++f) n[l.base_dcf + ((((size_t)c * O + o) * N + i) * L + e) * 4 + f] = "deltacc_front" + idx({c, o, i, e, f});
    }
    n[l.base_so + ((size_t)c * O + o) * N + i] = "slackvarsObstacle" + idx({c, o, i});
    for (int f = 0; f < 4; ++f) n[l.base_sof + (((size_t)c * O + o) * N + i) * 4 + f] = "slackvarsObstacle_front" + idx({c, o, i, f});
  }
  for (int a = 0; a < K; ++a) for (int b = 0; b < K; ++b) for (int i = 0; i < N; ++i) {
    for (int q = 0; q < 16; ++q) n[l.base_c2c + (((size_t)a * K + b) * N + i) * 16 + q] = "car2car_collision" + idx({a, b, i, q});
    for (int q = 0; q < 4; ++q) n[l.base_sv + (((size_t)a * K + b) * N + i) * 4 + q] = "slackvars" + idx({a, b, i, q});
  }
  return n;
}

bool WriteMst(const std::string &path, const MiqpB200Layout &l, const std::vector<double> &x) {
  if ((int)x.size() != l.ncols) return false;
  std::ofstream f(path);
  if (!f) return false;
  const std::vector<std::string> names = ColumnNames(l);
  f << "<?xml version = \"1.0\" encoding=\"UTF-8\" standalone=\"yes\"?>\n<CPLEXSolutions version=\"1.2\">\n <CPLEXSolution version=\"1.2\">\n"
    << "  <header\n    problemName=\"cplexmodel\"\n    solutionName=\"m1\"\n    solutionIndex=\"0\"\n    MIPStartEffortLevel=\"0\"\n    writeLevel=\"2\"/>\n  <variables>\n";
  f << std::setprecision(17);
  for (int k = 0; k < l.ncols; ++k) f << "   <variable name=\"" << names[k] << "\" index=\"" << k << "\" value=\"" << x[k] << "\"/>\n";
  f << "  </variables>\n </CPLEXSolution>\n</CPLEXSolutions>\n";
  return (bool)f;
}

bool ReadMst(const std::string &path, int ncols, std::vector<double> &x) {
  std::ifstream f(path);
  if (!f) return false;
  std::vector<double> v((size_t)ncols, 0.0);
  std::string line; int seen = 0;
  while (std::getline(f, line)) {
    const size_t pi = line.find("index=\""), pv = line.find("value=\"");
    if (line.find("<variable") == std::string::npos || pi == std::string::npos || pv == std::string::npos) continue;
    const int k = std::atoi(line.c_str() + pi + 7);
    if (k < 0 || k >= ncols) return false;
    v[k] = std::strtod(line.c_str() + pv + 7, nullptr);
    ++seen;
  }
  if (seen != ncols) return false;
  x.swap(v);
  return true;
}

bool B200Wrapper::writeMIPStarts(const std::string &mstfile) const { return haveLast_ && WriteMst(mstfile, lastLayout_, lastX_); }

bool B200Wrapper::readMIPStarts(const std::string &mstfile) {
  if (!parameters_) return false;
  FlatProblem fp; MiqpB200Layout l;
  try { Flatten(*parameters_, precision_, fp); } catch (const std::exception &) { return false; }
  if (miqp_b200_layout(&fp.p, &l) != MIQP_B200_OK) return false;
  std::vector<double> x;
  if (!ReadMst(mstfile, l.ncols, x)) return false;
  lastX_.swap(x); lastLayout_ = l; haveLast_ = true;
  return true;
}

bool B200Wrapper::exportModel(const std::string &lpfile) {
  error_.clear();
  if (!parameters_) { error_ = "resetParameters() has not been called"; return false; }
  FlatProblem fp; MiqpB200Layout l; MiqpB200Sizes sz;
  try { Flatten(*parameters_, source_ == DATFILE ? 0 : precision_, fp); } catch (const std::exception &ex) { error_ = ex.what(); return false; }
  if (miqp_b200_layout(&fp.p, &l) != MIQP_B200_OK) { error_ = "malformed ModelParameters"; return false; }
  if (!EnsureSolver()) return false;
  if (miqp_b200_sizes(solver_, &fp.p, &sz) != MIQP_B200_OK) { error_ = miqp_b200_last_error(solver_); return false; }
  std::vector<long> rowptr((size_t)sz.nrows + 1);
  std::vector<int> cols((size_t)sz.nnz_struct);
  std::vector<double> vals((size_t)sz.nnz_struct), lo((size_t)sz.nrows), hi((size_t)sz.nrows);
  if (miqp_b200_assemble(solver_, &fp.p, rowptr.data(), cols.data(), vals.data(), lo.data(), hi.data()) != MIQP_B200_OK) {
    error_ = miqp_b200_last_error(solver_); return false;
  }
  std::ofstream f(lpfile);
  if (!f) { error_ = "cannot write " + lpfile; return false; }
  const std::vector<std::string> names = ColumnNames(l);
  const MiqpB200Problem &p = fp.p;
  const int C = l.C, N = l.N;
  f << std::setprecision(15);
  f << "\\ENCODING=ISO-8859-1\n\\Problem name: cplexmodel\n\\ rows " << sz.nrows << ", non-zeros " << sz.nnz << ", columns " << l.ncols
    << " (" << sz.nbin << " binary)\n\nMinimize\n obj:";
  // objective_function.mod:7-19: sum w (v - ref)^2 + w a^2 + w u^2 + W_obs slackObs^2 + W_slack slackvars^2
  const double *w[8] = {p.w_jerk_x, p.w_jerk_y, p.w_pos_x, p.w_vel_x, p.w_acc_x, p.w_pos_y, p.w_vel_y, p.w_acc_y};   // per core block 0..7
  const double *ref[8] = {nullptr, nullptr, p.x_ref, p.vx_ref, nullptr, p.y_ref, p.vy_ref, nullptr};
  double konst = 0.0; int terms = 0;
  auto brk = [&]() { if (++terms % 6 == 0) f << "\n     "; };
  for (int b = 0; b < 8; ++b) for (int c = 0; c < C; ++c) for (int i = 0; i < N; ++i) {
    const double wt = w[b][c], r = ref[b] ? ref[b][(size_t)c * N + i] : 0.0;
    konst += wt * r * r;
    const double lin = -2.0 * wt * r;
    if (lin != 0.0) { f << (lin < 0 ? " - " : " + ") << std::fabs(lin) << " " << names[((size_t)b * C + c) * N + i]; brk(); }
  }
  f << " + " << konst << " objconst\n      + [";
  terms = 0;
  auto quad = [&](int col, double q) { if (q != 0.0) { f << " + " << 2.0 * q << " " << names[col] << " ^2"; brk(); } };
  for (int b = 0; b < 8; ++b) for (int c = 0; c < C; ++c) for (int i = 0; i < N; ++i) quad((b * C + c) * N + i, w[b][c]);
  for (int k = l.base_so; k < l.base_c2c; ++k) quad(k, p.w_slack_obs);
  for (int k = l.base_sv; k < l.ncols; ++k) quad(k, p.w_slack);
  f << " ] / 2\nSubject To\n";
  for (long r = 0; r < sz.nrows; ++r) {
    f << " c" << r + 1 << ":";
    int nt = 0;
    for (long k = rowptr[r]; k < rowptr[r + 1]; ++k) {
      if (vals[k] == 0.0) continue;
      f << (vals[k] < 0 ? " - " : " + ") << std::fabs(vals[k]) << " " << names[cols[k]];
      if (++nt % 5 == 0) f << "\n     ";
    }
    if (nt == 0) f << " 0 objconst";
    const bool flo = std::isfinite(lo[r]), fhi = std::isfinite(hi[r]);
    if (flo && fhi && lo[r] == hi[r]) f << " = " << lo[r];
    else if (fhi && !flo) f << " <= " << hi[r];
    else if (flo && !fhi) f << " >= " << lo[r];
    else { error_ = "ranged row in the model"; return false; }
    f << "\n";
  }
  f << "Bounds\n objconst = 1\n";
  for (int k = 0; k < l.base_nwe; ++k) f << " " << names[k] << " free\n";                         // decision_variables.mod:10-26
  for (int k = l.base_so; k < l.base_c2c; ++k) f << " 0 <= " << names[k] << " <= 1\n";            // :46-47
  for (int k = l.base_sv; k < l.ncols; ++k) f << " 0 <= " << names[k] << " <= " << p.maximum_slack << "\n";   // :53
  f << "Binaries\n";
  int nb = 0;
  for (int k = l.base_nwe; k < l.base_so; ++k) { f << " " << names[k]; if (++nb % 6 == 0) f << "\n"; }
  for (int k = l.base_c2c; k < l.base_sv; ++k) { f << " " << names[k]; if (++nb % 6 == 0) f << "\n"; }
  f << "\nEnd\n";
  return (bool)f;
}

void B200Wrapper::setDevice(int ordinal) {
  if (ordinal == device_) return;
  device_ = ordinal;
  if (solver_) { miqp_b200_destroy(solver_); solver_ = nullptr; }
}

void B200Wrapper::addRecedingHorizonWarmstart(std::shared_ptr<RawResults> warmstart, WarmstartType type) {
  useRecedingWarm_ = true;
  if (type != RECEDING_HORIZON_WARMSTART) useLastSolution_ = true;
  recedingWarm_ = warmstart;
}
void B200Wrapper::setLastSolutionWarmstart(WarmstartType type) {
  useLastSolution_ = true;
  if (type != LAST_SOLUTION_WARMSTART) useRecedingWarm_ = true;
}
void B200Wrapper::deleteLastSolutionWarmstartFile() { haveLast_ = false; std::remove(tmpWarmstartFile_.c_str()); }

bool B200Wrapper::EnsureSolver() {
  if (solver_) return true;
  MiqpB200Options opt; miqp_b200_default_options(&opt);
  opt.device = device_;
  if (miqp_b200_create(&opt, &solver_) != MIQP_B200_OK || !solver_) {
    solver_ = nullptr;
    error_ = "no usable CUDA device: the MIQP backend has no CPU fallback";
    return false;
  }
  return true;
}

bool B200Wrapper::setSolutionPoolCapacity(int capacity) {
  if (capacity < 0 || capacity > 64) return false;
  poolCapacity_ = capacity;
  return true;
}

bool B200Wrapper::getSolutionPoolResults(int j, RawResults &out) const {
  if (j < 0 || j >= (int)pool_.size()) return false;
  Unpack(poolLayout_, pool_[j].x.data(), out);
  return true;
}

// pool of plan k of the last run on `solver` (capacity poolCapacity_), best first; clears the pool when it is off
bool B200Wrapper::FetchPool(MiqpB200Solver *solver, int k, const MiqpB200Layout &layout) {
  pool_.clear();
  if (poolCapacity_ <= 0) return true;
  std::vector<MiqpB200PoolEntry> e(poolCapacity_);
  std::vector<double> x((size_t)poolCapacity_ * layout.ncols);
  int n = 0;
  if (miqp_b200_pool_fetch(solver, k, poolCapacity_, e.data(), x.data(), nullptr, &n) != MIQP_B200_OK) {
    const char *m = miqp_b200_last_error(solver);
    error_ = m ? m : "solution pool fetch failed";
    return false;
  }
  pool_.resize(n);
  for (int j = 0; j < n; ++j) {
    SolutionPoolEntry &o = pool_[j];
    o.objective = e[j].objective; o.max_violation = e[j].max_violation; o.converged = e[j].converged != 0;
    o.x.assign(x.begin() + (size_t)j * layout.ncols, x.begin() + (size_t)(j + 1) * layout.ncols);
  }
  poolLayout_ = layout;
  return true;
}

struct B200Wrapper::Prepared {
  FlatProblem flat;
  MiqpB200Layout layout{};
  std::vector<double> warm;
  bool have_warm = false;
};

bool B200Wrapper::Prepare(double timestamp, Prepared &pr) {
  error_.clear();
  if (source_ == DATFILE) {   // the file is the problem (fixtures, parameter dumps): no rounding on top of what was written
    try {
      if (!parameters_) parameters_ = std::make_shared<ModelParameters>();
      datio::ReadParametersDat(datFile_, *parameters_);
      Flatten(*parameters_, 0, pr.flat);
    } catch (const std::exception &ex) { error_ = ex.what(); return false; }
  } else {
    if (!parameters_) { error_ = "resetParameters() has not been called"; return false; }
    try { Flatten(*parameters_, precision_, pr.flat); } catch (const std::exception &ex) { error_ = ex.what(); return false; }
  }
  if (miqp_b200_layout(&pr.flat.p, &pr.layout) != MIQP_B200_OK) { error_ = "malformed ModelParameters"; return false; }
  pr.have_warm = false;
  if (useRecedingWarm_ && recedingWarm_ && recedingWarm_->NrCars == pr.layout.C && recedingWarm_->N == pr.layout.N &&
      recedingWarm_->NrRegions == pr.layout.R) {
    // the last column of every binary family is a repetition of the previous one (MiqpPlanner::CalculateWarmstart);
    // it is handed over as "undecided" so that the start is a partial assignment the search completes
    Pack(pr.layout, *recedingWarm_, true, pr.warm);
    pr.have_warm = true;
  } else if (useLastSolution_ && !haveLast_ && ReadMst(tmpWarmstartFile_, pr.layout.ncols, lastX_)) {
    // the MIP start of a previous solve (possibly by another wrapper or process) comes back from the warm-start file, as
    // in the reference (src/cplex_wrapper.cpp:128-138)
    lastLayout_ = pr.layout; haveLast_ = true;
    pr.warm = lastX_; pr.have_warm = true;
  } else if (useLastSolution_ && haveLast_ && lastLayout_.ncols == pr.layout.ncols && lastLayout_.C == pr.layout.C &&
             lastLayout_.E == pr.layout.E && lastLayout_.O == pr.layout.O) {
    pr.warm = lastX_; pr.have_warm = true;
  }
  if (!debugPath_.empty()) {
    std::ostringstream fn;
    fn << std::setprecision(15) << debugPath_ << "/" << debugPrefix_ << "parameters_" << timestamp << ".txt";
    if (WriteParametersDat(pr.flat.p, *parameters_, fn.str())) lastParameterFile_ = fn.str();
    if (debugPrint_) {   // lpexport_<t>.lp next to the parameter dump (src/cplex_wrapper.cpp:151-154)
      std::ostringstream ln;
      ln << std::setprecision(15) << debugPath_ << "/" << debugPrefix_ << "lpexport_" << timestamp << ".lp";
      exportModel(ln.str());
    }
  }
  return true;
}

OptimizationStatus B200Wrapper::Finish(const Prepared &pr, const MiqpB200SolveInfo &info, const double *x, double timestamp) {
  props_ = SolutionProperties();
  props_.time = info.seconds;
  props_.NrBinaryVariables = (pr.layout.base_so - pr.layout.base_nwe) + (pr.layout.base_sv - pr.layout.base_c2c);
  props_.NrFloatVariables = pr.layout.ncols - props_.NrBinaryVariables;
  props_.NrIterations = (int)info.qp_iters; props_.NrNodes = info.nodes; props_.NrRounds = info.rounds;
  props_.best_bound = info.best_bound;
  if (collectSizes_) {
    MiqpB200Sizes sz;
    if (miqp_b200_sizes(solver_, &pr.flat.p, &sz) == MIQP_B200_OK) { props_.NrConstraints = (int)sz.nrows; props_.NonZeroCoefficients = (int)sz.nnz; }
  }
  if (info.status == MIQP_B200_SUCCESS) {
    // CPLEX status codes callers may look at: 101 optimal, 102 optimal within tolerance, 107 time limit with incumbent
    props_.status = info.proven ? (info.gap == 0.0 ? 101 : 102) : 107;
    props_.objective = info.objective; props_.gap = info.gap; props_.max_violation = info.max_violation;
    props_.proven_gap = info.proven != 0; props_.NrSolutionPool = poolCapacity_ > 0 ? (int)pool_.size() : 1;
    Unpack(pr.layout, x, *results_);
    lastX_.assign(x, x + pr.layout.ncols); lastLayout_ = pr.layout; haveLast_ = true;
    if (useLastSolution_) WriteMst(tmpWarmstartFile_, lastLayout_, lastX_);   // cplex.writeMIPStarts, src/cplex_wrapper.cpp:206-209
    if (debugPrint_ && !debugPath_.empty()) {
      if (useLastSolution_) {
        std::ostringstream wn;
        wn << std::setprecision(15) << debugPath_ << "/" << debugPrefix_ << "warmstartsolution_" << timestamp << ".mst";
        WriteMst(wn.str(), lastLayout_, lastX_);
      }
      std::ostringstream fn;
      fn << std::setprecision(15) << debugPath_ << "/" << debugPrefix_ << "solution_" << timestamp << ".txt";
      std::ofstream f(fn.str());
      f << std::setprecision(12) << "// objective " << info.objective << " gap " << info.gap << " nodes " << info.nodes << "\n";
      static const char *names[12] = {"u_x", "u_y", "pos_x", "vel_x", "acc_x", "pos_y", "vel_y", "acc_y",
                                      "pos_x_front_UB", "pos_x_front_LB", "pos_y_front_UB", "pos_y_front_LB"};
      for (int b = 0; b < 12; ++b) {
        f << names[b] << " = [";
        for (int c = 0; c < pr.layout.C; ++c) {
          f << "[";
          for (int i = 0; i < pr.layout.N; ++i) f << (i ? " " : "") << x[((long)b * pr.layout.C + c) * pr.layout.N + i];
          f << "]";
        }
        f << "];\n";
      }
    }
    return SUCCESS;
  }
  props_.objective = NAN; props_.gap = NAN;
  pool_.clear();
  props_.status = (info.status == MIQP_B200_FAILED_TIMEOUT) ? 108 : 103;   // time limit without incumbent / integer infeasible
  return info.status == MIQP_B200_FAILED_TIMEOUT ? FAILED_TIMEOUT : FAILED_NO_SOLUT;
}

bool B200Wrapper::setSolutionVector(const double *x, int ncols) {
  if (!parameters_) return false;
  FlatProblem f;
  MiqpB200Layout l;
  try { Flatten(*parameters_, precision_, f); } catch (const std::exception &) { return false; }
  if (miqp_b200_layout(&f.p, &l) != MIQP_B200_OK || l.ncols != ncols) return false;
  Unpack(l, x, *results_);
  lastX_.assign(x, x + ncols); lastLayout_ = l; haveLast_ = true;
  return true;
}

OptimizationStatus B200Wrapper::callCplex(double timestamp) {
  Prepared pr;
  if (!Prepare(timestamp, pr)) return FAILED_SEG_FAULT;
  if (!EnsureSolver()) return FAILED_SEG_FAULT;
  std::vector<double> x(pr.layout.ncols, 0.0);
  const double *warm = pr.have_warm ? pr.warm.data() : nullptr;
  double *xo = x.data();
  MiqpB200SolveInfo info;
  pool_.clear();
  miqp_b200_set_solution_pool(solver_, poolCapacity_);   // (0..64: setSolutionPoolCapacity checked it)
  const int rc = miqp_b200_solve_batch(solver_, &pr.flat.p, 1, pr.have_warm ? &warm : nullptr, &xo, &info);
  if (rc != MIQP_B200_OK || (info.status == MIQP_B200_SUCCESS && !FetchPool(solver_, 0, pr.layout))) {
    const char *e = miqp_b200_last_error(solver_);
    error_ = e ? e : "device solve failed";
    props_ = SolutionProperties(); props_.objective = NAN; props_.gap = NAN;
    return FAILED_SEG_FAULT;
  }
  return Finish(pr, info, x.data(), timestamp);
}

long B200Wrapper::deviceWarmstartBatches_ = 0;

std::vector<OptimizationStatus> B200Wrapper::callBatch(const std::vector<B200Wrapper *> &solvers, double timestamp) {
  const int n = (int)solvers.size();
  std::vector<OptimizationStatus> out(n, FAILED_SEG_FAULT);
  if (n == 0) return out;
  std::vector<Prepared> pr(n);
  std::vector<int> idx;                      // solvers whose problem could be prepared
  for (int k = 0; k < n; ++k) if (solvers[k]->Prepare(timestamp, pr[k])) idx.push_back(k);
  if (idx.empty()) return out;
  B200Wrapper *lead = solvers[idx[0]];       // the batch runs on the first solver's device handle
  if (!lead->EnsureSolver()) { for (int k : idx) solvers[k]->error_ = lead->error_; return out; }
  const int m = (int)idx.size();
  std::vector<MiqpB200Problem> probs(m);
  std::vector<std::vector<double>> xs(m);
  std::vector<double *> xo(m);
  std::vector<const double *> warm(m, nullptr);
  bool any_warm = false;
  for (int j = 0; j < m; ++j) {
    const Prepared &p = pr[idx[j]];
    probs[j] = p.flat.p; xs[j].assign(p.layout.ncols, 0.0); xo[j] = xs[j].data();
    if (p.have_warm) { warm[j] = p.warm.data(); any_warm = true; }
  }
  std::vector<MiqpB200SolveInfo> infos(m);
  // Receding-horizon replanning of the same planners in the same order: the MIP starts are the previous incumbents, shifted by one
  // step on the device (miqp_b200_batch_upload_replan) -- the host-side shifted vectors (CalculateWarmstart) are not sent.
  std::vector<B200Wrapper *> members(m);
  bool all_warm = true;
  for (int j = 0; j < m; ++j) { members[j] = solvers[idx[j]]; all_warm = all_warm && pr[idx[j]].have_warm; }
  // solution pool: the batch keeps as many entries as its most demanding member asks for; each member takes its own share
  int pool_cap = 0;
  for (B200Wrapper *w : members) pool_cap = std::max(pool_cap, w->poolCapacity_);
  miqp_b200_set_solution_pool(lead->solver_, pool_cap);   // (0..64: setSolutionPoolCapacity checked it)
  int rc;
  if (lead->deviceWarmstart_ && all_warm && m > 1 && lead->lastBatch_ == members) {
    rc = miqp_b200_batch_upload_replan(lead->solver_, probs.data(), m);
    if (rc == MIQP_B200_OK) rc = miqp_b200_batch_run(lead->solver_, nullptr);
    if (rc == MIQP_B200_OK) rc = miqp_b200_batch_fetch(lead->solver_, xo.data(), infos.data());
    if (rc == MIQP_B200_OK) ++deviceWarmstartBatches_;
  } else {
    rc = miqp_b200_solve_batch(lead->solver_, probs.data(), m, any_warm ? warm.data() : nullptr, xo.data(), infos.data());
  }
  lead->lastBatch_ = (rc == MIQP_B200_OK) ? members : std::vector<B200Wrapper *>();
  if (rc != MIQP_B200_OK) {
    const char *e = miqp_b200_last_error(lead->solver_);
    for (int k : idx) solvers[k]->error_ = e ? e : "device solve failed";
    return out;
  }
  for (int j = 0; j < m; ++j) {   // before Finish: its model statistics (collectSizes_) replace the batch on the lead's handle
    B200Wrapper *w = solvers[idx[j]];
    if (infos[j].status == MIQP_B200_SUCCESS && !w->FetchPool(lead->solver_, j, pr[idx[j]].layout)) {
      out[idx[j]] = FAILED_SEG_FAULT;
      infos[j].status = -1;
    }
  }
  for (int j = 0; j < m; ++j) {
    B200Wrapper *w = solvers[idx[j]];
    if (infos[j].status == -1) continue;
    if (w->collectSizes_ && !w->EnsureSolver()) w->collectSizes_ = false;
    out[idx[j]] = w->Finish(pr[idx[j]], infos[j], xs[j].data(), timestamp);
  }
  return out;
}

}  // namespace cplex
}  // namespace planner
}  // namespace miqp
