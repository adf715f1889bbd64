// planner_data.hpp -- plain data contracts of the planner facade and the solver driver.
//
// Counterparts of the reference's src/miqp_planner_data.hpp: InitialStateIndices (:34-42),
// RawResults (:46-97), ModelParameters (:99-185), DefaultSettings / ApolloDefaultSettings
// (:190-251), plus SolutionProperties / OptimizationStatus of src/cplex_wrapper.hpp:41-59.
// Same member names and meaning, so code written against the reference structs reads the
// same; storage is the row-major containers of dense.hpp instead of Eigen.
//
// Quirk kept on purpose (SURVEY.md section C): RawResults stores the obstacle / agent slack
// variables, which are continuous in the model, in INT tensors, as the reference does
// (src/miqp_planner_data.hpp:88-92); the full-precision values stay available through
// B200Wrapper::getSolutionVector().
#pragma once
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/miqp_planner_settings.h"
#include "dense.hpp"

namespace miqp {
namespace planner {

using dense::MatrixXd;
using dense::MatrixXi;
using dense::VectorXd;
using dense::VectorXi;
template <class T, int R> using Tensor = dense::Tensor<T, R>;

enum InitialStateIndices : int {
  MIQP_STATE_X = 0, MIQP_STATE_VX = 1, MIQP_STATE_AX = 2,
  MIQP_STATE_Y = 3, MIQP_STATE_VY = 4, MIQP_STATE_AY = 5,
  MIQP_INITIAL_STATE_SIZE = 6
};

typedef unsigned int PolygonId;

struct LimitPerRegionParameters {   // [cars][regions]
  MatrixXd min_x, max_x, min_y, max_y;
};
struct PolynomialCurvatureParameters { MatrixXd POLY_KAPPA_AX_MAX, POLY_KAPPA_AX_MIN; };   // [R][3]
struct PolynomialOrientationParameters { MatrixXd POLY_SINT_UB, POLY_SINT_LB, POLY_COSS_UB, POLY_COSS_LB; };
typedef MatrixXd FractionParameters;   // [R][4]: x1 y1 x2 y2 of the two rays of a wedge

// one value per decision variable of cplexmodel/decision_variables.mod:10-53
struct RawResults {
  Tensor<double, 2> u_x, u_y, pos_x, vel_x, acc_x, pos_y, vel_y, acc_y;               // (NrCars, N)
  Tensor<double, 2> pos_x_front_UB, pos_x_front_LB, pos_y_front_UB, pos_y_front_LB;   // (NrCars, N)
  Tensor<int, 3> notWithinEnvironmentRear, notWithinEnvironmentFrontUbUb, notWithinEnvironmentFrontLbUb,
      notWithinEnvironmentFrontUbLb, notWithinEnvironmentFrontLbLb;                   // (NrCars, NrEnvironments, N)
  Tensor<int, 3> active_region;                                                       // (NrCars, N, NrRegions)
  Tensor<int, 2> region_change_not_allowed_x_positive, region_change_not_allowed_y_positive,
      region_change_not_allowed_x_negative, region_change_not_allowed_y_negative,
      region_change_not_allowed_combined;                                             // (NrCars, N)
  Tensor<int, 4> deltacc;             // (NrCars, NrObstacles, N, MaxLinesObstacles)
  Tensor<int, 5> deltacc_front;       // (NrCars, NrObstacles, N, MaxLinesObstacles, 4)
  Tensor<int, 4> car2car_collision;   // (K, K, N, 16), K = NrCars - 1
  Tensor<int, 4> slackvars;           // (K, K, N, 4)
  Tensor<int, 3> slackvarsObstacle;        // (NrCars, NrObstacles, N)
  Tensor<int, 4> slackvarsObstacle_front;  // (NrCars, NrObstacles, N, 4)
  int N = 0, NrEnvironments = 0, NrRegions = 0, NrObstacles = 0, MaxLinesObstacles = 0,
      NrCarToCarCollisions = 0, NrCars = 0;
};

struct ModelParameters {
  // solver parameters (cplexmodel/cplexmodel.mod:8-20).  Only the gap and the time limit steer
  // the device search; the CPLEX tuning knobs are carried for API compatibility.
  float max_solution_time = 10.f;
  float relative_mip_gap_tolerance = 0.1f;
  int mipdisplay = 2, mipemphasis = 0;
  float relobjdif = 0.f;
  int cutpass = 0, probe = 0, repairtries = 0, rinsheur = 0, varsel = 0, mircuts = 0, parallelmode = 0;
  // model parameters (cplexmodel/parameters.mod:8-136)
  int NumSteps = 0;
  float ts = 0.f;
  int nr_regions = 0;
  int NumCars = 0;
  float min_vel_x_y = 0.f, max_vel_x_y = 0.f;
  float total_min_acc = 0.f, total_max_acc = 0.f, total_min_jerk = 0.f, total_max_jerk = 0.f;
  VectorXd agent_safety_distance, agent_safety_distance_slack;   // [N]
  float maximum_slack = 0.f;
  VectorXd WEIGHTS_POS_X, WEIGHTS_VEL_X, WEIGHTS_ACC_X, WEIGHTS_POS_Y, WEIGHTS_VEL_Y, WEIGHTS_ACC_Y,
      WEIGHTS_JERK_X, WEIGHTS_JERK_Y;                            // [cars]
  float WEIGHTS_SLACK = 0.f, WEIGHTS_SLACK_OBSTACLE = 0.f;
  VectorXd WheelBase, CollisionRadius, BufferReference;          // [cars]
  MatrixXd IntitialState;                                        // (sic) [cars][6]
  MatrixXd x_ref, vx_ref, y_ref, vy_ref;                         // [cars][N]
  LimitPerRegionParameters acc_limit_params, jerk_limit_params;
  VectorXi initial_region;                                       // [cars], 1-based
  MatrixXi possible_region;                                      // [cars][R]
  int nr_obstacles = 0;
  std::vector<std::vector<MatrixXd>> ObstacleConvexPolygon;      // [obstacle][step] -> (k, 2) vertices
  int max_lines_obstacles = 0;
  std::vector<int> obstacle_is_soft;
  int nr_environments = 0;
  std::vector<MatrixXd> MultiEnvironmentConvexPolygon;           // (k, 2) vertices, counter-clockwise
  std::vector<PolygonId> environmentPolygonIds;
  FractionParameters fraction_parameters;
  float minimum_region_change_speed = 0.f;
  PolynomialCurvatureParameters poly_curvature_params;
  PolynomialOrientationParameters poly_orientation_params;
};

struct SolutionProperties {
  int status = 0;
  double gap = 0.0, objective = 0.0, time = 0.0;
  int NrConstraints = 0, NrBinaryVariables = 0, NrFloatVariables = 0, NonZeroCoefficients = 0;
  int NrIterations = 0;     // interior-point iterations summed over all node relaxations
  int NrSolutionPool = 0;   // entries of the solution pool (B200Wrapper::setSolutionPoolCapacity); with the pool off 1 if an incumbent exists
  // additions of the device search
  long NrNodes = 0, NrRounds = 0;
  double best_bound = 0.0, max_violation = 0.0;
  bool proven_gap = false;
};

enum OptimizationStatus { SUCCESS = 0, FAILED_NO_SOLUT = 1, FAILED_SEG_FAULT = 2, FAILED_TIMEOUT = 3 };

typedef MiqpPlannerSettings Settings;

inline Settings DefaultSettings() {
  Settings s;
  std::memset(&s, 0, sizeof s);
  s.nr_regions = 16; s.nr_steps = 20; s.nr_neighbouring_possible_regions = 1;
  s.ts = 0.25f; s.precision = 12;
  s.constant_agent_safety_distance_slack = 3.f; s.minimum_region_change_speed = 2.f;
  s.lambda = 0.5f; s.wheelBase = 2.8f; s.collisionRadius = 1.f;
  s.slackWeight = 30.f; s.slackWeightObstacle = 2000.f;
  s.jerkWeight = 1.f; s.positionWeight = 2.f; s.velocityWeight = 0.f; s.acclerationWeight = 0.f;
  s.accLonMaxLimit = 2.f; s.accLonMinLimit = -4.f; s.jerkLonMaxLimit = 3.f;
  s.accLatMinMaxLimit = 1.6f; s.jerkLatMinMaxLimit = 1.4f;
  s.simplificationDistanceMap = 0.2f; s.simplificationDistanceReferenceLine = 0.05f;
  s.bufferReference = s.collisionRadius; s.buffer_for_merging_tolerance = 0.1f;
  s.refLineInterpInc = 0.2f; s.additionalStepsForReferenceLongerHorizon = 4;
  s.max_solution_time = 10.f; s.relative_mip_gap_tolerance = 0.1f;
  s.mipdisplay = 2;   // mipemphasis .. mircuts stay 0
  std::strcpy(s.cplexModelpath, "cplexmodel/");
  s.useSos = false; s.useBranchingPriorities = false;
  s.warmstartType = NO_WARMSTART; s.parallelMode = AUTO;
  s.max_velocity_fitting = 20.f;
  s.buffer_cplex_outputs = false;
  s.obstacle_roi_filter = false;
  s.obstacle_roi_behind_distance = 5.f; s.obstacle_roi_front_distance = 30.f; s.obstacle_roi_side_distance = 15.f;
  return s;
}

inline Settings ApolloDefaultSettings() {
  Settings s = DefaultSettings();
  std::strcpy(s.cplexModelpath,
              "../bazel-bin/modules/planning/libplanning_component.so.runfiles/miqp_planner/cplex_modfiles/");
  s.buffer_cplex_outputs = true;
  return s;
}

}  // namespace planner
}  // namespace miqp
