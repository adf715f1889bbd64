// miqp_planner_c_api.cpp -- extern "C" shim over MiqpPlanner (include/miqp_planner_c_api.h).
// Same entry points and behaviour as the reference's src/miqp_planner_c_api.cpp:20-260.
#include "../../include/miqp_planner_c_api.h"
#include "../../include/miqp_planner_solution_pool.h"

#include <cassert>
#include <cmath>
#include <string>
#include <vector>

#include "miqp_planner.hpp"

using miqp::planner::MatrixXd;
using miqp::planner::MiqpPlanner;
using miqp::planner::Point2;
using miqp::planner::PolyLine;
using miqp::planner::RawResults;
using miqp::planner::RefPoint;

namespace {
inline MiqpPlanner *P(CMiqpPlanner h) { return reinterpret_cast<MiqpPlanner *>(h); }

// ConvertToBarkLine of the reference: points -> line, simplified with the given tolerance
PolyLine MakeLine(MiqpPlanner *p, const double *pts, int n, double tol) {
  std::vector<Point2> in(n), out;
  for (int k = 0; k < n; ++k) in[k] = {pts[2 * k], pts[2 * k + 1]};
  miqp::planner::SimplifyPolyline(in, tol, out);
  std::vector<double> flat;
  for (const Point2 &q : out) { flat.push_back(q.x); flat.push_back(q.y); }
  return PolyLine(flat.data(), (int)out.size(), p->GetSettings().refLineInterpInc);
}

std::vector<MatrixXd> Corners(const double *p1x, const double *p1y, const double *p2x, const double *p2y, const double *p3x,
                              const double *p3y, const double *p4x, const double *p4y, int size) {
  std::vector<MatrixXd> out;
  for (int i = 0; i < size; ++i) {
    MatrixXd o(4, 2);
    o(0, 0) = p1x[i]; o(0, 1) = p1y[i]; o(1, 0) = p2x[i]; o(1, 1) = p2y[i];
    o(2, 0) = p3x[i]; o(2, 1) = p3y[i]; o(3, 0) = p4x[i]; o(3, 1) = p4y[i];
    out.push_back(o);
  }
  return out;
}
}  // namespace

extern "C" {

CMiqpPlanner NewCMiqpPlanner() {
#if PLANNER_MIQP_CAPI_NO_APOLLO
  MiqpPlannerSettings s = miqp::planner::DefaultSettings();
#else
  MiqpPlannerSettings s = miqp::planner::ApolloDefaultSettings();
#endif
  return reinterpret_cast<void *>(new MiqpPlanner(s));
}

CMiqpPlanner NewCMiqpPlannerSettings(MiqpPlannerSettings settings) {
  try { return reinterpret_cast<void *>(new MiqpPlanner(settings)); }
  catch (const std::exception &) { return nullptr; }   // unknown (regions, vmax, vmin) table combination
}

void DelCMiqpPlanner(CMiqpPlanner h) { delete P(h); }

int AddCarCMiqpPlanner(CMiqpPlanner h, double initial_state_in[], double ref_in[], const int ref_size, double vDes,
                       double deltaSDes, const double timestep, const bool track_reference_positions) {
  const PolyLine line = MakeLine(P(h), ref_in, ref_size, P(h)->GetSettings().simplificationDistanceReferenceLine);
  return P(h)->AddCar(initial_state_in, line, vDes, deltaSDes, timestep, track_reference_positions);
}

bool PlanCMiqpPlanner(CMiqpPlanner h, const double timestep) { return P(h)->Plan(timestep); }

void UpdateCarCMiqpPlanner(CMiqpPlanner h, int idx, double initial_state_in[], double ref_in[], const int ref_size,
                           const double timestep, bool track_reference_positions) {
  const PolyLine line = MakeLine(P(h), ref_in, ref_size, P(h)->GetSettings().simplificationDistanceReferenceLine);
  P(h)->UpdateCar(idx, initial_state_in, line, timestep, track_reference_positions);
}

void ActivateDebugFileWriteCMiqpPlanner(CMiqpPlanner h, char path[], char name[]) {
  P(h)->ActivateDebugFileWrite(std::string(path), std::string(name));
}

int GetNCMiqpPlanner(CMiqpPlanner h) { return P(h)->GetN(); }
float GetTsCMiqpPlanner(CMiqpPlanner h) { return P(h)->GetTs(); }
float GetCollisionRadius(CMiqpPlanner h) { return P(h)->GetCollisionRadius(); }

void GetRawCMiqpTrajectoryCMiqpPlanner(CMiqpPlanner h, int carIdx, double start_time, double *trajectory, int &size) {
  const std::shared_ptr<RawResults> r = P(h)->GetSolution();
  assert(carIdx < r->NrCars);
  MiqpPlanner::RawTrajectoryRows(*r, carIdx, start_time, P(h)->GetParameters()->ts, trajectory, size);
}

void GetRawCLastReferenceTrajectoryCMiqpPlaner(CMiqpPlanner h, int carIdx, double start_time, double *trajectory, int &size) {
  const std::vector<RefPoint> &ref = P(h)->GetLastReference(carIdx);
  const float dt = P(h)->GetTs();
  const int N = P(h)->GetN();
  size = N;
  double time = start_time;
  for (int i = 0; i < N; ++i) {
    double *row = trajectory + (long)i * TRAJECTORY_SIZE;
    row[TRAJECTORY_TIME_IDX] = time;
    row[TRAJECTORY_X_IDX] = ref[i].x; row[TRAJECTORY_Y_IDX] = ref[i].y;
    row[TRAJECTORY_VX_IDX] = ref[i].v * std::cos(ref[i].theta); row[TRAJECTORY_VY_IDX] = ref[i].v * std::sin(ref[i].theta);
    row[TRAJECTORY_AX_IDX] = 0; row[TRAJECTORY_AY_IDX] = 0; row[TRAJECTORY_UX_IDX] = 0; row[TRAJECTORY_UY_IDX] = 0;   // not part of a reference
    time += dt;
  }
}

bool UpdateConvexifiedMapCMiqpPlaner(CMiqpPlanner h, double poly_pts[], const int poly_size) {
  std::vector<Point2> in(poly_size), out;
  for (int k = 0; k < poly_size; ++k) in[k] = {poly_pts[2 * k], poly_pts[2 * k + 1]};
  miqp::planner::SimplifyPolyline(in, P(h)->GetSettings().simplificationDistanceMap, out);
  MatrixXd poly((int)out.size(), 2);
  for (size_t k = 0; k < out.size(); ++k) { poly((int)k, 0) = out[k].x; poly((int)k, 1) = out[k].y; }
  return P(h)->UpdateConvexifiedMap(poly);
}

void UpdateDesiredVelocityCMiqpPlanner(CMiqpPlanner h, const int carIdx, const double vDes, const double deltaSDes) {
  P(h)->UpdateDesiredVelocity(carIdx, vDes, deltaSDes);
}

int AddObstacleCMiqpPlanner(CMiqpPlanner h, double p1_x[], double p1_y[], double p2_x[], double p2_y[], double p3_x[],
                            double p3_y[], double p4_x[], double p4_y[], const int size, bool is_static, bool is_soft) {
  std::vector<MatrixXd> o = Corners(p1_x, p1_y, p2_x, p2_y, p3_x, p3_y, p4_x, p4_y, size);
  return P(h)->AddObstacle(o, is_soft, is_static);
}

void UpdateObstacleCMiqpPlanner(CMiqpPlanner h, int id, double p1_x[], double p1_y[], double p2_x[], double p2_y[],
                                double p3_x[], double p3_y[], double p4_x[], double p4_y[], const int size, bool) {
  std::vector<MatrixXd> o = Corners(p1_x, p1_y, p2_x, p2_y, p3_x, p3_y, p4_x, p4_y, size);
  P(h)->UpdateObstacle(id, o);
}

void RemoveAllObstaclesCMiqpPlanner(CMiqpPlanner h) { P(h)->RemoveAllObstacles(); }

int PlanBatchCMiqpPlanner(CMiqpPlanner *planners, int count, const double timestep, bool *success) {
  std::vector<MiqpPlanner *> ps(count);
  for (int k = 0; k < count; ++k) ps[k] = P(planners[k]);
  const std::vector<bool> ok = MiqpPlanner::PlanBatch(ps, timestep);
  int n = 0;
  for (int k = 0; k < count; ++k) { if (success) success[k] = ok[k]; n += ok[k]; }
  return n;
}

bool SetSolutionPoolCapacityCMiqpPlanner(CMiqpPlanner h, int capacity) { return P(h)->SetSolutionPoolCapacity(capacity); }
int GetSolutionPoolSizeCMiqpPlanner(CMiqpPlanner h) { return P(h)->GetSolutionPoolSize(); }
double GetSolutionPoolTrajectoryCMiqpPlanner(CMiqpPlanner h, int j, int carIdx, double start_time, double *trajectory, int &size) {
  return P(h)->GetSolutionPoolTrajectory(j, carIdx, start_time, trajectory, size);
}

long DeviceWarmstartBatchesCMiqpPlanner() { return miqp::planner::cplex::B200Wrapper::deviceWarmstartBatches(); }

void GetSolutionPropertiesCMiqpPlanner(CMiqpPlanner h, double out[8]) {
  const miqp::planner::SolutionProperties s = P(h)->GetSolutionProperties();
  out[0] = s.objective; out[1] = s.gap; out[2] = s.time; out[3] = s.status; out[4] = (double)s.NrNodes;
  out[5] = s.NrConstraints; out[6] = s.NrBinaryVariables; out[7] = s.NrFloatVariables;
}

// test hooks: inject a solution vector (decision_variables.mod order) and read back the receding-horizon MIP start the
// planner derives from it (MiqpPlanner::CalculateWarmstart), packed into the same column order (NaN = undecided)
bool DebugSetSolutionCMiqpPlanner(CMiqpPlanner h, const double *x, int ncols) { return P(h)->GetCplexWrapper().setSolutionVector(x, ncols); }
int DebugWarmstartCMiqpPlanner(CMiqpPlanner h, double *out, int ncols, bool relax_last_step) {
  P(h)->RecomputeWarmstart();
  miqp::planner::cplex::FlatProblem f;
  MiqpB200Layout l;
  miqp::planner::cplex::Flatten(*P(h)->GetParameters(), P(h)->GetSettings().precision, f);
  if (miqp_b200_layout(&f.p, &l) != MIQP_B200_OK || l.ncols != ncols) return -1;
  std::vector<double> x;
  miqp::planner::cplex::Pack(l, *P(h)->GetWarmstart(), relax_last_step, x);
  for (int k = 0; k < ncols; ++k) out[k] = x[k];
  return ncols;
}

// test hook: the flattened problem of the planner's current ModelParameters, written as an OPL .dat file
bool DebugWriteParametersCMiqpPlanner(CMiqpPlanner h, const char *path, int initial_region_combination) {
  miqp::planner::cplex::FlatProblem f;
  (void)initial_region_combination;
  miqp::planner::cplex::Flatten(*P(h)->GetParameters(), P(h)->GetSettings().precision, f);
  return miqp::planner::cplex::WriteParametersDat(f.p, *P(h)->GetParameters(), path);
}

}  // extern "C"
