// miqp_planner.hpp -- planner facade over the B200 MIQP backend.
//
// Counterpart of the reference's MiqpPlanner (src/miqp_planner.hpp:27-432, src/miqp_planner.cpp):
// owns the ModelParameters of one joint plan (cars, obstacles, drivable area), prepares them
// on the CPU exactly as the reference does (AddCar/UpdateCar :180-390, obstacles :405-488,
// environment :490-537), and in Plan() (:633-766) loops over the start-region combinations
// around the solver call -- which here is the CUDA branch and bound behind B200Wrapper instead
// of CPLEX.  On success the receding-horizon MIP start of the next cycle is derived from the
// solution (CalculateWarmstart :787-1051, EnvironmentWarmstart :1053-1115).
//
// New: PlanBatch() plans many independent planners in ONE device batch (multi-scenario
// dispatch named by BASELINE.json:north_star).
//
// Geometry types: BARK / boost.geometry are not part of this build.  Reference lines are
// poly-lines (PolyLine), polygons are (k, 2) vertex matrices.  The drivable area may be given
// as a road polygon -- convex (shrunk by the collision radius, one cell) or non-convex
// (decomposed by host/convexified_map.hpp: ear clipping + Hertel-Mehlhorn merging, boundary
// edges moved inwards; the reference: common/map/convexified_map.cpp) -- or as a ready convex
// decomposition (SetConvexEnvironmentCells).  A polygon that cannot be decomposed makes
// UpdateConvexifiedMap return false and Plan() refuse to run (fail closed).
#pragma once
#include <array>
#include <cmath>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "b200_wrapper.hpp"
#include "planner_data.hpp"
#include "planner_prep.hpp"

namespace miqp {
namespace planner {

class NotImplementedException : public std::logic_error {
 public:
  NotImplementedException() : std::logic_error{"Function not yet implemented."} {}
};

class MiqpPlanner {
 public:
  MiqpPlanner();
  explicit MiqpPlanner(const Settings &settings);
  MiqpPlanner(const Settings &settings, const MatrixXd &mapPolygon);
  // copies share parameters_ and warmstart_ and get a fresh solver (reference src/miqp_planner.cpp:153-175)
  MiqpPlanner(const MiqpPlanner &o);

  // initialState = {x, vx, ax, y, vy, ay}; returns the car index (0 = ego)
  int AddCar(const double initialState[6], const PolyLine &referencePath, double desiredVelocity,
             double deltaSForDesiredVel, double timestep = 0.0, bool track_reference_positions = true);
  void UpdateCar(int idx, const double initialState[6], const PolyLine &referencePath, double timestep = 0.0,
                 bool track_reference_positions = true);
  void RemoveCar(int idx);
  void UpdateDesiredVelocity(int carIdx, double vDes, double deltaSDes);

  // one (k, 2) vertex matrix per time step; -1 if the obstacle touches neither drivable area nor region of interest
  int AddObstacle(std::vector<MatrixXd> &dynamic_obstacle, bool is_soft, bool is_static);
  // box obstacle from predicted poses (x, y, theta per step; one pose = static), inflated by the
  // collision radius as CreateMiqpObstacle does
  int AddObstacle(const std::vector<std::array<double, 3>> &poses, double length, double width, bool is_soft, bool is_static);
  std::vector<MatrixXd> CreateMiqpObstacle(const std::vector<std::array<double, 3>> &poses, double length, double width) const;
  void UpdateObstacle(int id, std::vector<MatrixXd> &dynamic_obstacle);
  void RemoveObstacle(int id);        // throws NotImplementedException, like the reference
  void RemoveAllObstacles();

  bool UpdateConvexifiedMap(const MatrixXd &mapPolygon);                 // convex or non-convex road polygon (see above)
  void SetConvexEnvironmentCells(const std::vector<MatrixXd> &cells);   // already shrunk, convex, any orientation

  bool Plan(double timestamp = 0.0);
  static std::vector<bool> PlanBatch(const std::vector<MiqpPlanner *> &planners, double timestamp = 0.0);

  std::shared_ptr<RawResults> GetSolution() const { return cplexWrapper_.getRawResults(); }
  // Solution pool of every Plan() / PlanBatch(): up to `capacity` (0..64, 0 = off) best distinct feasible plans, entry 0 = the
  // solution Plan() returned.  GetSolutionPoolTrajectory fills rows like GetRawCMiqpTrajectoryCMiqpPlanner and returns the
  // entry's objective (NaN and size 0 if there is no entry j).
  bool SetSolutionPoolCapacity(int capacity) { return cplexWrapper_.setSolutionPoolCapacity(capacity); }
  int GetSolutionPoolSize() const { return (int)cplexWrapper_.getSolutionPool().size(); }
  double GetSolutionPoolTrajectory(int j, int carIdx, double start_time, double *trajectory, int &size) const;
  SolutionProperties GetSolutionProperties() const { return cplexWrapper_.getSolutionProperties(); }
  const cplex::B200Wrapper &GetCplexWrapper() const { return cplexWrapper_; }
  cplex::B200Wrapper &GetCplexWrapper() { return cplexWrapper_; }
  std::shared_ptr<ModelParameters> GetParameters() { return parameters_; }
  std::shared_ptr<RawResults> GetWarmstart() const { return warmstart_; }
  bool HasValidWarmstart() const { return validWarmstart_; }
  const Settings &GetSettings() const { return settings_; }
  int GetN() const { return settings_.nr_steps; }
  float GetTs() const { return settings_.ts; }
  float GetCollisionRadius() const { return settings_.collisionRadius; }
  int GetNrCars() const { return parameters_->NumCars; }
  const std::vector<RefPoint> &GetLastReference(int carIdx) const { return referenceGenerator_.at(carIdx).GetLastTrajectory(); }
  void ActivateDebugFileWrite(const std::string &path, const std::string &name);
  void SetDoWarmstart(MiqpPlannerWarmstartType in) { doWarmstart_ = in; }
  // receding-horizon MIP start from the solution the solver currently holds (what Plan() does after a success)
  void RecomputeWarmstart() { CalculateWarmstart(); }
  // state {x, vx, ax, y, vy, ay} of the plan at step timeIdx (Get2ndOrderStateFromSolution / GetThirdOrderStateAtResultIdx)
  void Get2ndOrderStateFromSolution(int timeIdx, int carIdx, double out[6]) const;
  // Plan of one car as rows {t, x, y, theta, v} (the reference's GetBarkTrajectory, src/miqp_planner.cpp:1132-1170):
  // theta = atan2(vy, vx), v = |(vx, vy)|; the trajectory is cut at the first step whose |vx| and |vy| are both
  // <= 0.7 m/s, where the heading is no longer defined.
  std::vector<std::array<double, 5>> GetTrajectory(int carIdx, double start_time) const;
  static bool IsVxVyValid(double vx, double vy) { return std::fabs(vx) > 0.7 || std::fabs(vy) > 0.7; }
  // {x, y, theta, v, a} -> {x, vx, ax, y, vy, ay}, in float like the reference (src/miqp_planner.cpp:1189-1199)
  static void CarStateToMiqpState(float x, float y, float theta, float v, float a, double out[6]);
  // rows {t, x, y, vx, vy, ax, ay, ux, uy} of car carIdx (TRAJECTORY_* of the planner C ABI), N rows from start_time in steps of dt
  static void RawTrajectoryRows(const RawResults &r, int carIdx, double start_time, float dt, double *trajectory, int &size);

 private:
  struct PlanContext { std::vector<std::vector<int>> combos; size_t next = 0; std::vector<char> rollback; bool ready = false; };
  bool BeginPlan(PlanContext &ctx);                 // regions, environment, start pose check
  bool NextCombination(PlanContext &ctx);           // sets initial_region / possible_region, MIP start
  void RollbackCombination(PlanContext &ctx);
  bool EndPlan(OptimizationStatus status);
  void ResetEnvironment();
  void CalculateWarmstart();
  void EnvironmentWarmstart();
  bool ObstacleIntersectsEnvironment(const std::vector<MatrixXd> &obstacle, bool is_static) const;
  void UpdateObstaclesROI(double x, double y, double theta);
  void RecomputeTotalLimits();

  std::shared_ptr<ModelParameters> parameters_;
  std::shared_ptr<RawResults> warmstart_;
  MiqpPlannerWarmstartType doWarmstart_;
  bool validWarmstart_ = false;
  std::vector<PolygonId> environmentIdsWarmstart_;
  Settings settings_;
  ParameterPreparer parameterPreparer_;
  int egoCarIdx_ = 0;
  std::vector<ReferenceTrajectoryGenerator> referenceGenerator_, referenceGeneratorLongerHorizon_;
  bool mapRejected_ = false;                        // the last UpdateConvexifiedMap failed: Plan() returns false until a map is accepted
  std::vector<MatrixXd> mapCells_;                  // convex, CCW, shrunk by the collision radius; id = index
  std::map<PolygonId, MatrixXd> activeCells_;       // cells touched by the buffered references in the last Plan()
  MatrixXd mapPolygon_;
  MatrixXd obstaclesRoi_;
  cplex::B200Wrapper cplexWrapper_;
  const double eps_ = 1e-6;
};

}  // namespace planner
}  // namespace miqp
