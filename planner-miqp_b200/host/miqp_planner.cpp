// miqp_planner.cpp -- see miqp_planner.hpp.  Reference: src/miqp_planner.cpp.
#include "miqp_planner.hpp"
#include "convexified_map.hpp"
#include "../../include/miqp_planner_c_api.h"   // TRAJECTORY_* row layout

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>

namespace miqp {
namespace planner {

using cplex::B200Wrapper;

static const float kEps = 0.000001f;   // reference src/miqp_planner.hpp:415

MiqpPlanner::MiqpPlanner() : MiqpPlanner(DefaultSettings(), MatrixXd()) {}
MiqpPlanner::MiqpPlanner(const Settings &settings) : MiqpPlanner(settings, MatrixXd()) {}

MiqpPlanner::MiqpPlanner(const Settings &settings, const MatrixXd &mapPolygon)
    : parameters_(std::make_shared<ModelParameters>()),
      warmstart_(std::make_shared<RawResults>()),
      doWarmstart_(settings.warmstartType),
      settings_(settings),
      parameterPreparer_(settings.nr_regions, settings.max_velocity_fitting, settings.minimum_region_change_speed,
                         settings.accLonMaxLimit, settings.accLonMinLimit, settings.jerkLonMaxLimit,
                         settings.accLatMinMaxLimit, settings.jerkLatMinMaxLimit),
      cplexWrapper_(settings.cplexModelpath, "cplexmodel.mod", B200Wrapper::CPPINPUTS, settings.precision) {
  cplexWrapper_.resetParameters(parameters_);
  cplexWrapper_.deleteLastSolutionWarmstartFile();
  ModelParameters &p = *parameters_;
  p.nr_regions = settings.nr_regions; p.NumSteps = settings.nr_steps;
  p.NumCars = 0; p.nr_obstacles = 0; p.nr_environments = 0; p.max_lines_obstacles = 0;
  const FittingTableSet &t = parameterPreparer_.Tables();
  const int R = settings.nr_regions;
  p.poly_orientation_params.POLY_SINT_UB = TableToMatrix(t.t[0], R);
  p.poly_orientation_params.POLY_SINT_LB = TableToMatrix(t.t[1], R);
  p.poly_orientation_params.POLY_COSS_UB = TableToMatrix(t.t[2], R);
  p.poly_orientation_params.POLY_COSS_LB = TableToMatrix(t.t[3], R);
  p.poly_curvature_params.POLY_KAPPA_AX_MAX = TableToMatrix(t.t[4], R);
  p.poly_curvature_params.POLY_KAPPA_AX_MIN = TableToMatrix(t.t[5], R);
  p.max_solution_time = settings.max_solution_time;
  p.relative_mip_gap_tolerance = settings.relative_mip_gap_tolerance;
  p.mipdisplay = settings.mipdisplay; p.mipemphasis = settings.mipemphasis; p.relobjdif = settings.relobjdif;
  p.cutpass = settings.cutpass; p.probe = settings.probe; p.repairtries = settings.repairtries;
  p.rinsheur = settings.rinsheur; p.varsel = settings.varsel; p.mircuts = settings.mircuts;
  p.parallelmode = (int)settings.parallelMode;
  p.ts = settings.ts;
  p.minimum_region_change_speed = settings.minimum_region_change_speed;
  p.agent_safety_distance.resize(p.NumSteps);
  p.agent_safety_distance_slack.resize(p.NumSteps);
  p.agent_safety_distance_slack.setConstant(settings.constant_agent_safety_distance_slack);
  p.maximum_slack = settings.constant_agent_safety_distance_slack;
  p.WEIGHTS_SLACK = settings.slackWeight; p.WEIGHTS_SLACK_OBSTACLE = settings.slackWeightObstacle;
  p.min_vel_x_y = -settings.max_velocity_fitting - kEps;
  p.max_vel_x_y = +settings.max_velocity_fitting + kEps;
  p.fraction_parameters = parameterPreparer_.GetFractionParameters();
  if (mapPolygon.rows() >= 3) UpdateConvexifiedMap(mapPolygon);
  warmstart_->N = settings_.nr_steps; warmstart_->NrRegions = settings_.nr_regions;
  cplexWrapper_.setSpecialOrderedSets(settings.useSos);
  cplexWrapper_.setUseBranchingPriorities(settings.useBranchingPriorities);
  cplexWrapper_.setBranchingPriorityValueExtent(1, settings_.nr_steps - 1);
  if (settings_.buffer_cplex_outputs) cplexWrapper_.setBufferCplexOutputsToStream(true);
}

MiqpPlanner::MiqpPlanner(const MiqpPlanner &o)
    : parameters_(o.parameters_), warmstart_(o.warmstart_), doWarmstart_(o.doWarmstart_), validWarmstart_(o.validWarmstart_),
      environmentIdsWarmstart_(o.environmentIdsWarmstart_), settings_(o.settings_), parameterPreparer_(o.parameterPreparer_),
      egoCarIdx_(o.egoCarIdx_), referenceGenerator_(o.referenceGenerator_),
      referenceGeneratorLongerHorizon_(o.referenceGeneratorLongerHorizon_), mapCells_(o.mapCells_), activeCells_(o.activeCells_),
      mapPolygon_(o.mapPolygon_), obstaclesRoi_(o.obstaclesRoi_), cplexWrapper_(o.cplexWrapper_) {
  mapRejected_ = o.mapRejected_;
  cplexWrapper_.resetParameters(parameters_);
}

void MiqpPlanner::RecomputeTotalLimits() {
  ModelParameters &p = *parameters_;
  p.total_max_acc = std::max(p.acc_limit_params.max_x.maxCoeff(), p.acc_limit_params.max_y.maxCoeff()) + kEps;
  p.total_min_acc = std::min(p.acc_limit_params.min_x.minCoeff(), p.acc_limit_params.min_y.minCoeff()) - kEps;
  p.total_max_jerk = std::max(p.jerk_limit_params.max_x.maxCoeff(), p.jerk_limit_params.max_y.maxCoeff()) + kEps;
  p.total_min_jerk = std::min(p.jerk_limit_params.min_x.minCoeff(), p.jerk_limit_params.min_y.minCoeff()) - kEps;
}

int MiqpPlanner::AddCar(const double initialState[6], const PolyLine &referencePath, double desiredVelocity,
                        double deltaSForDesiredVel, double timestep, bool track_reference_positions) {
  ModelParameters &p = *parameters_;
  const int idx = p.NumCars, n = idx + 1, N = settings_.nr_steps, R = p.nr_regions;
  p.NumCars = n;
  p.CollisionRadius.conservativeResize(n); p.CollisionRadius(idx) = settings_.collisionRadius;
  p.WheelBase.conservativeResize(n); p.WheelBase(idx) = settings_.wheelBase;
  p.IntitialState.conservativeResize(n, MIQP_INITIAL_STATE_SIZE);
  std::vector<double> acc[4], jerk[4];
  parameterPreparer_.AccLimits(acc); parameterPreparer_.JerkLimits(jerk);
  MatrixXd *am[4] = {&p.acc_limit_params.min_x, &p.acc_limit_params.max_x, &p.acc_limit_params.min_y, &p.acc_limit_params.max_y};
  MatrixXd *jm[4] = {&p.jerk_limit_params.min_x, &p.jerk_limit_params.max_x, &p.jerk_limit_params.min_y, &p.jerk_limit_params.max_y};
  for (int k = 0; k < 4; ++k) {
    am[k]->conservativeResize(n, R); am[k]->setRow(idx, acc[k].begin());
    jm[k]->conservativeResize(n, R); jm[k]->setRow(idx, jerk[k].begin());
  }
  RecomputeTotalLimits();
  p.x_ref.conservativeResize(n, N); p.y_ref.conservativeResize(n, N);
  p.vx_ref.conservativeResize(n, N); p.vy_ref.conservativeResize(n, N);
  referenceGenerator_.emplace_back(settings_.ts, N, settings_.refLineInterpInc, desiredVelocity, deltaSForDesiredVel);
  referenceGeneratorLongerHorizon_.emplace_back(settings_.ts, N + settings_.additionalStepsForReferenceLongerHorizon,
                                                settings_.refLineInterpInc, desiredVelocity, deltaSForDesiredVel);
  p.possible_region.conservativeResize(n, R);
  p.initial_region.conservativeResize(n);
  VectorXd *w[8] = {&p.WEIGHTS_POS_X, &p.WEIGHTS_VEL_X, &p.WEIGHTS_ACC_X, &p.WEIGHTS_POS_Y,
                    &p.WEIGHTS_VEL_Y, &p.WEIGHTS_ACC_Y, &p.WEIGHTS_JERK_X, &p.WEIGHTS_JERK_Y};
  for (VectorXd *v : w) v->conservativeResize(n);
  UpdateCar(idx, initialState, referencePath, timestep, track_reference_positions);
  validWarmstart_ = false;   // sizes changed
  return idx;
}

void MiqpPlanner::UpdateCar(int idx, const double s[6], const PolyLine &referencePath, double, bool track) {
  ModelParameters &p = *parameters_;
  const int N = settings_.nr_steps, R = p.nr_regions;
  for (int k = 0; k < 6; ++k) p.IntitialState(idx, k) = s[k];
  const double theta = std::atan2(s[MIQP_STATE_VY], s[MIQP_STATE_VX]);
  const double v0 = std::sqrt(s[MIQP_STATE_VX] * s[MIQP_STATE_VX] + s[MIQP_STATE_VY] * s[MIQP_STATE_VY]);
  const std::vector<RefPoint> &ref = referenceGenerator_.at(idx).Generate(s[MIQP_STATE_X], s[MIQP_STATE_Y], theta, v0, referencePath);
  for (int i = 0; i < N; ++i) {
    p.x_ref(idx, i) = ref[i].x; p.y_ref(idx, i) = ref[i].y;
    p.vx_ref(idx, i) = ref[i].v * std::cos(ref[i].theta);
    p.vy_ref(idx, i) = ref[i].v * std::sin(ref[i].theta);
  }
  // possible regions: every wedge the headings of the (longer) reference pass through, widened
  const std::vector<RefPoint> &lref = referenceGeneratorLongerHorizon_.at(idx).Generate(s[MIQP_STATE_X], s[MIQP_STATE_Y], theta, v0, referencePath);
  for (int j = 0; j < R; ++j) p.possible_region(idx, j) = 0;
  for (const RefPoint &q : lref)
    for (int j : CalculateRegionIdx(p.fraction_parameters, (float)std::cos(q.theta), (float)std::sin(q.theta))) p.possible_region(idx, j) = 1;
  if (!ReserveNeighborRegions(p.possible_region, idx, settings_.nr_neighbouring_possible_regions))
    std::fprintf(stderr, "[miqp_planner] region expansion failed for car %d\n", idx);
  // weights: ego gets lambda, the others share 1 - lambda
  double scale;
  if (idx == egoCarIdx_) scale = settings_.lambda;
  else scale = (1 - settings_.lambda) / (p.NumCars - 1);
  if (track) {
    p.WEIGHTS_POS_X(idx) = scale * settings_.positionWeight; p.WEIGHTS_VEL_X(idx) = scale * settings_.velocityWeight;
    p.WEIGHTS_POS_Y(idx) = scale * settings_.positionWeight; p.WEIGHTS_VEL_Y(idx) = scale * settings_.velocityWeight;
  } else {
    p.WEIGHTS_POS_X(idx) = 0; p.WEIGHTS_VEL_X(idx) = 2; p.WEIGHTS_POS_Y(idx) = 0; p.WEIGHTS_VEL_Y(idx) = 2;
  }
  p.WEIGHTS_ACC_X(idx) = scale * settings_.acclerationWeight; p.WEIGHTS_ACC_Y(idx) = scale * settings_.acclerationWeight;
  p.WEIGHTS_JERK_X(idx) = scale * settings_.jerkWeight; p.WEIGHTS_JERK_Y(idx) = scale * settings_.jerkWeight;
  if (settings_.obstacle_roi_filter && idx == egoCarIdx_) UpdateObstaclesROI(s[MIQP_STATE_X], s[MIQP_STATE_Y], theta);
}

void MiqpPlanner::RemoveCar(int idx) {
  ModelParameters &p = *parameters_;
  if (idx == egoCarIdx_) { std::fprintf(stderr, "[miqp_planner] cannot remove the ego vehicle (idx %d)\n", idx); return; }
  if (idx >= p.NumCars) { std::fprintf(stderr, "[miqp_planner] no vehicle with idx %d\n", idx); return; }
  if (idx != p.NumCars - 1) throw NotImplementedException();   // only the last car can go, as in the reference
  const int n = p.NumCars - 1, N = settings_.nr_steps, R = settings_.nr_regions;
  p.NumCars = n;
  p.CollisionRadius.conservativeResize(n); p.WheelBase.conservativeResize(n);
  p.IntitialState.conservativeResize(n, MIQP_INITIAL_STATE_SIZE);
  MatrixXd *lm[8] = {&p.acc_limit_params.min_x, &p.acc_limit_params.max_x, &p.acc_limit_params.min_y, &p.acc_limit_params.max_y,
                     &p.jerk_limit_params.min_x, &p.jerk_limit_params.max_x, &p.jerk_limit_params.min_y, &p.jerk_limit_params.max_y};
  for (MatrixXd *m : lm) m->conservativeResize(n, R);
  p.x_ref.conservativeResize(n, N); p.y_ref.conservativeResize(n, N); p.vx_ref.conservativeResize(n, N); p.vy_ref.conservativeResize(n, N);
  p.possible_region.conservativeResize(n, R); p.initial_region.conservativeResize(n);
  VectorXd *w[8] = {&p.WEIGHTS_POS_X, &p.WEIGHTS_VEL_X, &p.WEIGHTS_ACC_X, &p.WEIGHTS_POS_Y,
                    &p.WEIGHTS_VEL_Y, &p.WEIGHTS_ACC_Y, &p.WEIGHTS_JERK_X, &p.WEIGHTS_JERK_Y};
  for (VectorXd *v : w) v->conservativeResize(n);
  referenceGenerator_.erase(referenceGenerator_.begin() + idx);
  referenceGeneratorLongerHorizon_.erase(referenceGeneratorLongerHorizon_.begin() + idx);
  RecomputeTotalLimits();
  validWarmstart_ = false;
}

void MiqpPlanner::UpdateDesiredVelocity(int carIdx, double vDes, double deltaSDes) {
  referenceGenerator_.at(carIdx).ResetDesiredVelocity(vDes, deltaSDes);
  referenceGeneratorLongerHorizon_.at(carIdx).ResetDesiredVelocity(vDes, deltaSDes);
}

// ---------------------------------------------------------------------------------------
int MiqpPlanner::AddObstacle(std::vector<MatrixXd> &dynamic_obstacle, bool is_soft, bool is_static) {
  if (!ObstacleIntersectsEnvironment(dynamic_obstacle, is_static)) return -1;
  ModelParameters &p = *parameters_;
  p.ObstacleConvexPolygon.push_back(dynamic_obstacle);
  p.obstacle_is_soft.push_back((int)is_soft);
  p.nr_obstacles = (int)p.ObstacleConvexPolygon.size();
  p.max_lines_obstacles = 4;   // rectangles
  validWarmstart_ = false;
  return p.nr_obstacles - 1;
}

std::vector<MatrixXd> MiqpPlanner::CreateMiqpObstacle(const std::vector<std::array<double, 3>> &poses, double length, double width) const {
  std::vector<MatrixXd> out;
  const double hl = length / 2.0 + settings_.collisionRadius, hw = width / 2.0 + settings_.collisionRadius;
  const double cx[4] = {-hl, hl, hl, -hl}, cy[4] = {-hw, -hw, hw, hw};   // counter-clockwise, no repeated closing vertex
  for (int i = 0; i < settings_.nr_steps; ++i) {
    const std::array<double, 3> &q = poses[std::min<size_t>(i, poses.size() - 1)];
    const double c = std::cos(q[2]), s = std::sin(q[2]);
    MatrixXd v(4, 2);
    for (int k = 0; k < 4; ++k) { v(k, 0) = q[0] + c * cx[k] - s * cy[k]; v(k, 1) = q[1] + s * cx[k] + c * cy[k]; }
    out.push_back(v);
  }
  return out;
}

int MiqpPlanner::AddObstacle(const std::vector<std::array<double, 3>> &poses, double length, double width, bool is_soft, bool is_static) {
  if (poses.empty()) return -1;
  std::vector<MatrixXd> o = CreateMiqpObstacle(poses, length, width);
  return AddObstacle(o, is_soft, is_static);
}

void MiqpPlanner::UpdateObstacle(int id, std::vector<MatrixXd> &dynamic_obstacle) { parameters_->ObstacleConvexPolygon.at(id) = dynamic_obstacle; }
void MiqpPlanner::RemoveObstacle(int) { throw NotImplementedException(); }
void MiqpPlanner::RemoveAllObstacles() {
  ModelParameters &p = *parameters_;
  p.ObstacleConvexPolygon.clear(); p.obstacle_is_soft.clear();
  p.nr_obstacles = 0; p.max_lines_obstacles = 0;
  validWarmstart_ = false;
}

bool MiqpPlanner::ObstacleIntersectsEnvironment(const std::vector<MatrixXd> &obstacle, bool is_static) const {
  if (mapCells_.empty()) return true;   // empty environment: keep every obstacle
  for (const MatrixXd &o : obstacle) {
    if (obstaclesRoi_.rows() >= 3 && !ConvexIntersect(obstaclesRoi_, o)) {
      if (is_static) return false;       // a static obstacle outside the region of interest never matters
      continue;
    }
    if (!activeCells_.empty()) { for (const auto &c : activeCells_) if (ConvexIntersect(c.second, o)) return true; }
    else for (const MatrixXd &c : mapCells_) if (ConvexIntersect(c, o)) return true;
  }
  return false;
}

void MiqpPlanner::UpdateObstaclesROI(double x, double y, double theta) {
  // rectangle around the ego pose in the ego frame; same corner arithmetic as the reference (src/miqp_planner.cpp:1308-1336)
  const double b = settings_.obstacle_roi_behind_distance, f = settings_.obstacle_roi_front_distance, w = settings_.obstacle_roi_side_distance;
  const double fx = x + std::cos(theta) * f, fy = y + std::sin(theta) * f;
  const double rx = x + std::cos(theta + M_PI) * b, ry = y + std::sin(theta + M_PI) * b;
  obstaclesRoi_.resize(4, 2);
  obstaclesRoi_(0, 0) = fx + std::sin(theta) * w; obstaclesRoi_(0, 1) = fy + std::cos(theta) * w;
  obstaclesRoi_(1, 0) = fx - std::sin(theta) * w; obstaclesRoi_(1, 1) = fy - std::cos(theta) * w;
  obstaclesRoi_(2, 0) = rx - std::sin(theta) * w; obstaclesRoi_(2, 1) = ry - std::cos(theta) * w;
  obstaclesRoi_(3, 0) = rx + std::sin(theta) * w; obstaclesRoi_(3, 1) = ry + std::cos(theta) * w;
}

// ---------------------------------------------------------------------------------------
bool MiqpPlanner::UpdateConvexifiedMap(const MatrixXd &polygon) {
  if (polygon == mapPolygon_ && !mapCells_.empty()) return true;   // unchanged map: keep the decomposition
  MatrixXd v = polygon;
  // drop a repeated closing vertex, orient counter-clockwise (Polygon2MiqpPolygonDefinition, common/geometry/geometry.cpp:126-139)
  if (v.rows() >= 2 && v(0, 0) == v(v.rows() - 1, 0) && v(0, 1) == v(v.rows() - 1, 1)) {
    MatrixXd t(v.rows() - 1, 2);
    for (int k = 0; k < t.rows(); ++k) { t(k, 0) = v(k, 0); t(k, 1) = v(k, 1); }
    v = t;
  }
  if (v.rows() < 3) return false;
  if (SignedArea(v) < 0) v = Reversed(v);
  // convex polygons are one cell; non-convex ones are decomposed into convex cells whose boundary edges are moved inwards
  // by the collision radius (host/convexified_map.hpp; the reference: ConvexifiedMap::Convert, common/map/convexified_map.cpp:60-128)
  miqp::common::map::ConvexifiedMap cm(v, settings_.collisionRadius, settings_.simplificationDistanceMap, settings_.bufferReference);
  if (!cm.Convert()) {
    // fail closed: without a valid decomposition Plan() refuses to run instead of planning without road boundaries
    std::fprintf(stderr, "[miqp_planner] the map polygon could not be decomposed into convex cells (degenerate, self-intersecting "
                         "or narrower than twice the collision radius)\n");
    mapCells_.clear(); activeCells_.clear(); mapRejected_ = true;
    return false;
  }
  mapPolygon_ = polygon;
  mapCells_.clear();
  for (const auto &kv : cm.GetMapConvexPolygons()) mapCells_.push_back(kv.second);
  activeCells_.clear();
  mapRejected_ = false;
  return true;
}

void MiqpPlanner::SetConvexEnvironmentCells(const std::vector<MatrixXd> &cells) {
  mapCells_.clear(); activeCells_.clear(); mapRejected_ = false;
  for (MatrixXd v : cells) {
    if (v.rows() < 3) continue;
    if (SignedArea(v) < 0) v = Reversed(v);
    mapCells_.push_back(v);
  }
  mapPolygon_ = MatrixXd();
}

void MiqpPlanner::ResetEnvironment() {
  ModelParameters &p = *parameters_;
  activeCells_.clear();
  for (const ReferenceTrajectoryGenerator &g : referenceGeneratorLongerHorizon_) {
    std::vector<Point2> pts;
    for (const RefPoint &q : g.GetLastTrajectory()) pts.push_back({q.x, q.y});
    for (size_t id = 0; id < mapCells_.size(); ++id)
      if (LineBufferTouchesConvex(pts, settings_.bufferReference, mapCells_[id])) activeCells_[(PolygonId)id] = mapCells_[id];
  }
  p.MultiEnvironmentConvexPolygon.clear(); p.environmentPolygonIds.clear();
  for (const auto &c : activeCells_) { p.MultiEnvironmentConvexPolygon.push_back(c.second); p.environmentPolygonIds.push_back(c.first); }
  p.nr_environments = (int)p.MultiEnvironmentConvexPolygon.size();
  if (validWarmstart_) EnvironmentWarmstart();
}

// ---------------------------------------------------------------------------------------
bool MiqpPlanner::BeginPlan(PlanContext &ctx) {
  if (mapRejected_) {
    std::fprintf(stderr, "[miqp_planner] the last map update was rejected: not planning without an environment\n");
    return false;
  }
  ModelParameters &p = *parameters_;
  ctx = PlanContext();
  if (p.NumCars <= 0) return false;
  std::vector<std::vector<int>> per_car(p.NumCars);
  for (int c = 0; c < p.NumCars; ++c) {
    per_car[c] = CalculateRegionIdx(parameterPreparer_.GetFractionParameters(), (float)p.IntitialState(c, MIQP_STATE_VX),
                                    (float)p.IntitialState(c, MIQP_STATE_VY));
    if (per_car[c].empty()) return false;
  }
  CalculateRegionCombinations(per_car, {}, ctx.combos);
  if (!mapCells_.empty()) {
    ResetEnvironment();
    for (int c = 0; c < p.NumCars; ++c) {   // start pose (rear and front axle) must lie in some cell
      const double x = p.IntitialState(c, 0), y = p.IntitialState(c, 3);
      const double th = std::atan2(p.IntitialState(c, 4), p.IntitialState(c, 1));
      const double fx = x + std::cos(th) * p.WheelBase(c), fy = y + std::sin(th) * p.WheelBase(c);
      bool rear = false, front = false;
      for (const auto &cell : activeCells_) { rear |= PointInConvex(cell.second, x, y); front |= PointInConvex(cell.second, fx, fy); }
      if (!rear || !front) { std::fprintf(stderr, "[miqp_planner] initial pose of car %d collides (%s axle)\n", c, rear ? "front" : "rear"); return false; }
    }
  }
  ctx.rollback.assign(p.NumCars, 0);
  ctx.ready = true;
  return true;
}

bool MiqpPlanner::NextCombination(PlanContext &ctx) {
  if (!ctx.ready || ctx.next >= ctx.combos.size()) return false;
  ModelParameters &p = *parameters_;
  const std::vector<int> &combo = ctx.combos[ctx.next++];
  for (int c = 0; c < p.NumCars; ++c) {
    p.initial_region(c) = combo[c] + 1;          // 1-based, as the OPL model indexes regions
    if (p.possible_region(c, combo[c]) == 0) { p.possible_region(c, combo[c]) = 1; ctx.rollback[c] = 1; }
    else ctx.rollback[c] = 0;
  }
  if ((doWarmstart_ == RECEDING_HORIZON_WARMSTART || doWarmstart_ == BOTH_WARMSTART_STRATEGIES) && validWarmstart_)
    cplexWrapper_.addRecedingHorizonWarmstart(warmstart_, doWarmstart_);
  if (doWarmstart_ == LAST_SOLUTION_WARMSTART || doWarmstart_ == BOTH_WARMSTART_STRATEGIES)
    cplexWrapper_.setLastSolutionWarmstart(doWarmstart_);
  return true;
}

void MiqpPlanner::RollbackCombination(PlanContext &ctx) {
  ModelParameters &p = *parameters_;
  for (int c = 0; c < p.NumCars; ++c)
    if (ctx.rollback[c]) p.possible_region(c, p.initial_region(c) - 1) = 0;
}

bool MiqpPlanner::EndPlan(OptimizationStatus status) {
  validWarmstart_ = false;
  if (status != SUCCESS) return false;
  if (doWarmstart_ == RECEDING_HORIZON_WARMSTART || doWarmstart_ == BOTH_WARMSTART_STRATEGIES) CalculateWarmstart();
  return true;
}

bool MiqpPlanner::Plan(double timestamp) {
  PlanContext ctx;
  if (!BeginPlan(ctx)) return false;
  OptimizationStatus status = FAILED_NO_SOLUT;
  while (NextCombination(ctx)) {
    status = cplexWrapper_.callCplex(timestamp);
    if (status == SUCCESS) break;
    if (status == FAILED_SEG_FAULT || status == FAILED_TIMEOUT) {
      std::fprintf(stderr, "[miqp_planner] optimisation failed (status %d) %s\n", (int)status, cplexWrapper_.lastError().c_str());
      return false;
    }
    RollbackCombination(ctx);
  }
  return EndPlan(status);
}

std::vector<bool> MiqpPlanner::PlanBatch(const std::vector<MiqpPlanner *> &planners, double timestamp) {
  const size_t n = planners.size();
  std::vector<bool> ok(n, false);
  std::vector<PlanContext> ctx(n);
  std::vector<size_t> live;
  for (size_t k = 0; k < n; ++k) if (planners[k]->BeginPlan(ctx[k]) && planners[k]->NextCombination(ctx[k])) live.push_back(k);
  while (!live.empty()) {
    std::vector<B200Wrapper *> solvers;
    for (size_t k : live) solvers.push_back(&planners[k]->cplexWrapper_);
    const std::vector<OptimizationStatus> st = B200Wrapper::callBatch(solvers, timestamp);
    std::vector<size_t> again;
    for (size_t j = 0; j < live.size(); ++j) {
      const size_t k = live[j];
      if (st[j] == SUCCESS) { ok[k] = planners[k]->EndPlan(SUCCESS); continue; }
      if (st[j] == FAILED_NO_SOLUT) {          // try the next start-region combination in the next batch
        planners[k]->RollbackCombination(ctx[k]);
        if (planners[k]->NextCombination(ctx[k])) { again.push_back(k); continue; }
      }
      planners[k]->EndPlan(st[j]);
    }
    live.swap(again);
  }
  return ok;
}

// ---------------------------------------------------------------------------------------
void MiqpPlanner::CalculateWarmstart() {
  const std::shared_ptr<RawResults> rr = cplexWrapper_.getRawResults();
  RawResults &w = *warmstart_;
  const int N = rr->N, C = rr->NrCars, E = rr->NrEnvironments, R = rr->NrRegions, K = rr->NrCarToCarCollisions,
            L = rr->MaxLinesObstacles, O = rr->NrObstacles;
  w = *rr;   // same shapes; every family is then shifted one step to the left
  const double ts = parameters_->ts;
  const double vm = parameters_->minimum_region_change_speed;
  Tensor<double, 2> *cont[12] = {&w.u_x, &w.u_y, &w.pos_x, &w.vel_x, &w.acc_x, &w.pos_y, &w.vel_y, &w.acc_y,
                                 &w.pos_x_front_UB, &w.pos_x_front_LB, &w.pos_y_front_UB, &w.pos_y_front_LB};
  for (Tensor<double, 2> *t : cont) for (int c = 0; c < C; ++c) for (int i = 0; i + 1 < N; ++i) (*t)(c, i) = (*t)(c, i + 1);
  Tensor<int, 2> *rc[5] = {&w.region_change_not_allowed_x_positive, &w.region_change_not_allowed_y_positive,
                           &w.region_change_not_allowed_x_negative, &w.region_change_not_allowed_y_negative,
                           &w.region_change_not_allowed_combined};
  for (Tensor<int, 2> *t : rc) for (int c = 0; c < C; ++c) for (int i = 0; i + 1 < N; ++i) (*t)(c, i) = (*t)(c, i + 1);
  for (int c = 0; c < C; ++c) {
    // last column: one forward-Euler step from the (shifted) column before it
    w.u_x(c, N - 1) = 0.0; w.u_y(c, N - 1) = 0.0;
    w.pos_x(c, N - 1) = w.pos_x(c, N - 2) + ts * w.vel_x(c, N - 2);
    w.pos_y(c, N - 1) = w.pos_y(c, N - 2) + ts * w.vel_y(c, N - 2);
    w.vel_x(c, N - 1) = w.vel_x(c, N - 2) + ts * w.acc_x(c, N - 2);
    w.vel_y(c, N - 1) = w.vel_y(c, N - 2) + ts * w.acc_y(c, N - 2);
    w.acc_x(c, N - 1) = w.acc_x(c, N - 2) + ts * w.u_x(c, N - 2);
    w.acc_y(c, N - 1) = w.acc_y(c, N - 2) + ts * w.u_y(c, N - 2);
    w.pos_x_front_UB(c, N - 1) = w.pos_x_front_UB(c, N - 2) + ts * w.vel_x(c, N - 2);
    w.pos_x_front_LB(c, N - 1) = w.pos_x_front_LB(c, N - 2) + ts * w.vel_x(c, N - 2);
    w.pos_y_front_UB(c, N - 1) = w.pos_y_front_UB(c, N - 2) + ts * w.vel_y(c, N - 2);
    w.pos_y_front_LB(c, N - 1) = w.pos_y_front_LB(c, N - 2) + ts * w.vel_y(c, N - 2);
    const int xp = w.vel_x(c, N - 1) <= vm, yp = w.vel_y(c, N - 1) <= vm, xn = w.vel_x(c, N - 1) >= -vm, yn = w.vel_y(c, N - 1) >= -vm;
    w.region_change_not_allowed_x_positive(c, N - 1) = xp; w.region_change_not_allowed_y_positive(c, N - 1) = yp;
    w.region_change_not_allowed_x_negative(c, N - 1) = xn; w.region_change_not_allowed_y_negative(c, N - 1) = yn;
    w.region_change_not_allowed_combined(c, N - 1) = (xp + yp + xn + yn) > 3;
  }
  Tensor<int, 3> *nwe[5] = {&w.notWithinEnvironmentRear, &w.notWithinEnvironmentFrontUbUb, &w.notWithinEnvironmentFrontLbUb,
                            &w.notWithinEnvironmentFrontUbLb, &w.notWithinEnvironmentFrontLbLb};
  for (Tensor<int, 3> *t : nwe) for (int c = 0; c < C; ++c) for (int e = 0; e < E; ++e) for (int i = 0; i + 1 < N; ++i) (*t)(c, e, i) = (*t)(c, e, i + 1);
  // active region: shifted; the last step is the wedge of the final velocity
  for (int c = 0; c < C; ++c) {
    for (int i = 0; i + 1 < N; ++i) for (int j = 0; j < R; ++j) w.active_region(c, i, j) = w.active_region(c, i + 1, j);
    for (int j = 0; j < R; ++j) w.active_region(c, N - 1, j) = 0;
    const std::vector<int> reg = CalculateRegionIdx(parameterPreparer_.GetFractionParameters(), (float)rr->vel_x(c, N - 1), (float)rr->vel_y(c, N - 1));
    if (!reg.empty()) w.active_region(c, N - 1, reg.front()) = 1;
  }
  for (int a = 0; a < K; ++a) for (int b = 0; b < K; ++b) for (int i = 0; i + 1 < N; ++i) {
    for (int q = 0; q < 16; ++q) w.car2car_collision(a, b, i, q) = w.car2car_collision(a, b, i + 1, q);
    for (int q = 0; q < 4; ++q) w.slackvars(a, b, i, q) = w.slackvars(a, b, i + 1, q);
  }
  for (int c = 0; c < C; ++c) for (int o = 0; o < O; ++o) for (int i = 0; i + 1 < N; ++i) for (int l = 0; l < L; ++l) {
    w.deltacc(c, o, i, l) = w.deltacc(c, o, i + 1, l);
    for (int q = 0; q < 4; ++q) w.deltacc_front(c, o, i, l, q) = w.deltacc_front(c, o, i + 1, l, q);
  }
  environmentIdsWarmstart_ = parameters_->environmentPolygonIds;
  validWarmstart_ = true;
}

// the set of active environment cells changed between two cycles: re-index the environment binaries
void MiqpPlanner::EnvironmentWarmstart() {
  const ModelParameters &p = *parameters_;
  if (p.environmentPolygonIds == environmentIdsWarmstart_) return;
  RawResults &w = *warmstart_;
  const int N = p.NumSteps, C = p.NumCars, E = p.nr_environments;
  Tensor<int, 3> *nwe[5] = {&w.notWithinEnvironmentRear, &w.notWithinEnvironmentFrontUbUb, &w.notWithinEnvironmentFrontLbUb,
                            &w.notWithinEnvironmentFrontUbLb, &w.notWithinEnvironmentFrontLbLb};
  for (Tensor<int, 3> *t : nwe) {
    const Tensor<int, 3> last = *t;
    t->resize(C, E, N);
    t->setConstant(1);   // "not in this cell" unless known from the last run
    for (int c = 0; c < C && c < last.dimension(0); ++c)
      for (int e = 0; e < E; ++e) {
        const auto it = std::find(environmentIdsWarmstart_.begin(), environmentIdsWarmstart_.end(), p.environmentPolygonIds[e]);
        if (it == environmentIdsWarmstart_.end()) continue;
        const int from = (int)(it - environmentIdsWarmstart_.begin());
        if (from >= last.dimension(1)) continue;
        for (int i = 0; i + 1 < N; ++i) (*t)(c, e, i) = last(c, from, i);
      }
  }
  w.NrEnvironments = E;
  environmentIdsWarmstart_ = p.environmentPolygonIds;
}

void MiqpPlanner::ActivateDebugFileWrite(const std::string &path, const std::string &name) {
  cplexWrapper_.setDebugOutputFilePath(path);
  cplexWrapper_.setDebugOutputFilePrefix(name);
  cplexWrapper_.setDebugOutputPrint(true);
}

void MiqpPlanner::Get2ndOrderStateFromSolution(int i, int c, double out[6]) const {
  const std::shared_ptr<RawResults> r = cplexWrapper_.getRawResults();
  out[0] = r->pos_x(c, i); out[1] = r->vel_x(c, i); out[2] = r->acc_x(c, i);
  out[3] = r->pos_y(c, i); out[4] = r->vel_y(c, i); out[5] = r->acc_y(c, i);
}

std::vector<std::array<double, 5>> MiqpPlanner::GetTrajectory(int c, double start_time) const {
  const std::shared_ptr<RawResults> r = cplexWrapper_.getRawResults();
  std::vector<std::array<double, 5>> out;
  const float dt = parameters_->ts;
  for (int i = 0; i < r->N; ++i) {
    const double vx = r->vel_x(c, i), vy = r->vel_y(c, i);
    if (!IsVxVyValid(vx, vy)) break;   // heading undefined from here on
    out.push_back({start_time + i * dt, r->pos_x(c, i), r->pos_y(c, i), std::atan2(vy, vx), std::sqrt(vx * vx + vy * vy)});
  }
  return out;
}

void MiqpPlanner::RawTrajectoryRows(const RawResults &r, int carIdx, double start_time, float dt, double *trajectory, int &size) {
  const int N = r.N;
  size = N;
  double time = start_time;
  for (int i = 0; i < N; ++i) {
    double *row = trajectory + (long)i * TRAJECTORY_SIZE;
    row[TRAJECTORY_TIME_IDX] = time;
    row[TRAJECTORY_X_IDX] = r.pos_x(carIdx, i); row[TRAJECTORY_Y_IDX] = r.pos_y(carIdx, i);
    row[TRAJECTORY_VX_IDX] = r.vel_x(carIdx, i); row[TRAJECTORY_VY_IDX] = r.vel_y(carIdx, i);
    row[TRAJECTORY_AX_IDX] = r.acc_x(carIdx, i); row[TRAJECTORY_AY_IDX] = r.acc_y(carIdx, i);
    row[TRAJECTORY_UX_IDX] = r.u_x(carIdx, i); row[TRAJECTORY_UY_IDX] = r.u_y(carIdx, i);
    time += dt;
  }
}

double MiqpPlanner::GetSolutionPoolTrajectory(int j, int carIdx, double start_time, double *trajectory, int &size) const {
  RawResults r;
  size = 0;
  if (!cplexWrapper_.getSolutionPoolResults(j, r) || carIdx < 0 || carIdx >= r.NrCars) return NAN;
  RawTrajectoryRows(r, carIdx, start_time, parameters_->ts, trajectory, size);
  return cplexWrapper_.getSolutionPool()[j].objective;
}

void MiqpPlanner::CarStateToMiqpState(float x, float y, float theta, float v, float a, double out[6]) {
  out[MIQP_STATE_X] = (double)x; out[MIQP_STATE_Y] = (double)y;
  out[MIQP_STATE_VX] = (double)(std::cos(theta) * v); out[MIQP_STATE_VY] = (double)(std::sin(theta) * v);
  out[MIQP_STATE_AX] = (double)(std::cos(theta) * a); out[MIQP_STATE_AY] = (double)(std::sin(theta) * a);
}

}  // namespace planner
}  // namespace miqp
