// python_module.cpp -- pybind11 module `miqp`: the Python surface of the reference's test module
// (python/bindings/python_module.cpp:13-20: CplexWrapper, SolutionProperties, OptimizationStatus, WarmstartType,
// ParallelMode, ConvexifiedMap) over the B200 host classes.  Built by planner-miqp_b200/build.py:build_pymodule().
//
// Differences that a caller sees: ConvexifiedMap takes the road polygon as an (n, 2) array and the reference line as an
// (n, 2) array of x, y (or a BARK trajectory array: columns 1 and 2 are x and y) instead of BARK geometry objects; its first
// argument (the BARK parameter server) is accepted and ignored.  BehaviorMiqpAgent (bound inside BARK's own module in the
// reference, python/bindings/python_planner_miqp.cpp) is bound here in its BARK-free form (host/behavior_miqp_agent.hpp): the
// observed world is a dict of plain arrays, the parameter server a dict with the reference's "Miqp::..." names.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "b200_wrapper.hpp"
#include "behavior_miqp_agent.hpp"
#include "convexified_map.hpp"

namespace py = pybind11;
using miqp::common::map::ConvexifiedMap;
using miqp::planner::MatrixXd;
using miqp::planner::OptimizationStatus;
using miqp::planner::SolutionProperties;
using miqp::planner::cplex::CplexWrapper;

namespace {

MatrixXd to_matrix(const py::array_t<double, py::array::c_style | py::array::forcecast> &a) {
  if (a.ndim() != 2 || a.shape(1) < 2) throw std::invalid_argument("expected an (n, 2) array of x, y");
  MatrixXd m((int)a.shape(0), 2);
  auto r = a.unchecked<2>();
  for (py::ssize_t k = 0; k < a.shape(0); ++k) { m((int)k, 0) = r(k, 0); m((int)k, 1) = r(k, 1); }
  return m;
}
py::array_t<double> to_array(const MatrixXd &m) {
  py::array_t<double> a({(py::ssize_t)m.rows(), (py::ssize_t)2});
  auto w = a.mutable_unchecked<2>();
  for (int k = 0; k < m.rows(); ++k) { w(k, 0) = m(k, 0); w(k, 1) = m(k, 1); }
  return a;
}
py::dict to_dict(const miqp::common::map::PolygonMap &pm) {
  py::dict d;
  for (const auto &kv : pm) d[py::int_(kv.first)] = to_array(kv.second);
  return d;
}

}  // namespace

PYBIND11_MODULE(miqp, m) {
  m.doc() = "B200-native MIQP planner backend: Python surface of planner-miqp's `miqp` test module";

  py::class_<ConvexifiedMap, std::shared_ptr<ConvexifiedMap>>(m, "ConvexifiedMap")
      .def(py::init([](py::object /*params*/, const py::array_t<double, py::array::c_style | py::array::forcecast> &poly, double buffer_radius,
                       double max_simplify_dist, double buffer_reference, double buffer_for_merging_tolerance) {
             return std::make_shared<ConvexifiedMap>(to_matrix(poly), buffer_radius, max_simplify_dist, buffer_reference, buffer_for_merging_tolerance);
           }),
           py::arg("params"), py::arg("map_polygon"), py::arg("buffer_radius"), py::arg("max_simplify_dist"), py::arg("buffer_reference"),
           py::arg("buffer_for_merging_tolerance"))
      .def("Convert", &ConvexifiedMap::Convert)
      .def("GetIntersectingConvexPolygons",
           [](const ConvexifiedMap &cm, const py::array_t<double, py::array::c_style | py::array::forcecast> &ref) {
             if (ref.ndim() != 2 || ref.shape(1) < 2) throw std::invalid_argument("expected an (n, 2) array of x, y or a BARK trajectory array");
             const int cx = ref.shape(1) >= 3 ? 1 : 0, cy = cx + 1;   // BARK StateDefinition: TIME, X, Y, THETA, VEL
             std::vector<miqp::planner::Point2> pts;
             auto r = ref.unchecked<2>();
             for (py::ssize_t k = 0; k < ref.shape(0); ++k) pts.push_back({r(k, cx), r(k, cy)});
             return to_dict(cm.GetIntersectingConvexPolygons(pts));
           })
      .def("HasValidPolygon", &ConvexifiedMap::HasValidPolygon)
      .def_property_readonly("map_nonconvex_polygon", [](const ConvexifiedMap &cm) { return to_array(cm.GetMapNonConvexPolygon()); }, "input map polygon.")
      .def_property_readonly("map_convex_polygons", [](const ConvexifiedMap &cm) { return to_dict(cm.GetMapConvexPolygons()); }, "decomposed convex polygons.");

  py::class_<CplexWrapper>(m, "CplexWrapper")
      // (modfile, precision): the reference's shorthand for a solver that reads an OPL .dat file (src/cplex_wrapper.hpp:119-120)
      .def(py::init([](const char *modfile, int precision) { return new CplexWrapper("cplexmodel/", modfile, CplexWrapper::DATFILE, precision); }))
      .def("setParameterDatFileAbsolute", &CplexWrapper::setParameterDatFileAbsolute)
      .def("callCplex", &CplexWrapper::callCplex, py::arg("timestamp") = 0.0, py::call_guard<py::gil_scoped_release>())
      .def("setDebugOutputFilePath", &CplexWrapper::setDebugOutputFilePath)
      .def("setDebugOutputFilePrefix", &CplexWrapper::setDebugOutputFilePrefix)
      .def("setDebugOutputPrint", &CplexWrapper::setDebugOutputPrint)
      .def("getDebugOutputParameterFilePath", &CplexWrapper::getDebugOutputParameterFilePath)
      .def("getSolutionProperties", &CplexWrapper::getSolutionProperties)
      // beyond the reference's binding: the file formats of the solver class
      .def("exportModel", &CplexWrapper::exportModel)
      .def("writeMIPStarts", &CplexWrapper::writeMIPStarts)
      .def("readMIPStarts", &CplexWrapper::readMIPStarts)
      .def("lastError", &CplexWrapper::lastError)
      .def("getSolutionVector", [](const CplexWrapper &w) { const std::vector<double> &x = w.getSolutionVector(); return py::array_t<double>(x.size(), x.data()); })
      // solution pool: up to `capacity` best distinct feasible plans of every solve, best first (entry 0 = the solution)
      .def("setSolutionPoolCapacity", &CplexWrapper::setSolutionPoolCapacity)
      .def("getSolutionPool", [](const CplexWrapper &w) {
        py::list out;
        for (const miqp::planner::cplex::SolutionPoolEntry &e : w.getSolutionPool())
          out.append(py::make_tuple(e.objective, e.max_violation, e.converged, py::array_t<double>(e.x.size(), e.x.data())));
        return out;
      }, "list of (objective, max_violation, converged, full column vector)");

  // ---- BehaviorMiqpAgent (src/behavior_miqp_agent.cpp:37-335) -------------------------------------------------------------
  using miqp::planner::BehaviorMiqpAgent;
  using miqp::planner::BehaviorStatus;
  using miqp::planner::ObservedAgent;
  using miqp::planner::ObservedWorldLite;
  py::enum_<BehaviorStatus>(m, "BehaviorStatus")
      .value("NOT_STARTED_YET", BehaviorStatus::NOT_STARTED_YET)
      .value("VALID", BehaviorStatus::VALID)
      .value("EXPIRED", BehaviorStatus::EXPIRED);
  auto agent_from = [](const py::dict &d) {
    ObservedAgent a;
    if (d.contains("id")) a.id = d["id"].cast<int>();
    const std::vector<double> st = d["state"].cast<std::vector<double>>();     // x, y, theta, v [, a]
    if (st.size() < 4) throw std::invalid_argument("agent state = [x, y, theta, v] or [x, y, theta, v, a]");
    a.x = st[0]; a.y = st[1]; a.theta = st[2]; a.v = st[3]; a.a = st.size() > 4 ? st[4] : 0.0;
    if (d.contains("length")) a.length = d["length"].cast<double>();
    if (d.contains("width")) a.width = d["width"].cast<double>();
    const auto lc = d["lane_center"].cast<py::array_t<double, py::array::c_style | py::array::forcecast>>();
    if (lc.ndim() != 2 || lc.shape(1) != 2 || lc.shape(0) < 2) throw std::invalid_argument("lane_center: (n, 2) array of x, y, n >= 2");
    auto r = lc.unchecked<2>();
    for (py::ssize_t k = 0; k < lc.shape(0); ++k) { a.lane_center.push_back(r(k, 0)); a.lane_center.push_back(r(k, 1)); }
    if (d.contains("prediction")) {
      const auto pr = d["prediction"].cast<py::array_t<double, py::array::c_style | py::array::forcecast>>();
      if (pr.ndim() != 2 || pr.shape(1) != 3) throw std::invalid_argument("prediction: (n, 3) array of x, y, theta");
      auto q = pr.unchecked<2>();
      for (py::ssize_t k = 0; k < pr.shape(0); ++k) a.prediction.push_back({q(k, 0), q(k, 1), q(k, 2)});
    }
    return a;
  };
  py::class_<BehaviorMiqpAgent>(m, "BehaviorMiqpAgent")
      .def(py::init([](const py::dict &params) {
             miqp::planner::Settings s = miqp::planner::DefaultSettings();
             BehaviorMiqpAgent::Params q;
             auto num = [&](const char *k, auto &dst) { if (params.contains(k)) dst = params[k].cast<std::decay_t<decltype(dst)>>(); };
             // planner settings (src/miqp_settings_from_param_server.hpp) and agent parameters, reference names
             num("Miqp::NrRegions", s.nr_regions); num("Miqp::NrSteps", s.nr_steps); num("Miqp::Ts", s.ts);
             num("Miqp::MaxSolutionTime", s.max_solution_time); num("Miqp::RelativeMIPGapTolerance", s.relative_mip_gap_tolerance);
             num("Miqp::CollisionRadius", s.collisionRadius); num("Miqp::WheelBase", s.wheelBase);
             num("Miqp::SlackWeight", s.slackWeight); num("Miqp::JerkWeight", s.jerkWeight); num("Miqp::PositionWeight", s.positionWeight);
             num("Miqp::VelocityWeight", s.velocityWeight); num("Miqp::MaxVelocityFitting", s.max_velocity_fitting);
             num("Miqp::MinimumRegionChangeSpeed", s.minimum_region_change_speed);
             if (params.contains("Miqp::WarmstartType")) s.warmstartType = (MiqpPlannerWarmstartType)params["Miqp::WarmstartType"].cast<int>();
             num("Miqp::DesiredVelocity", q.desired_velocity); num("Miqp::DeltaSDesiredVelocity", q.delta_s_desired_velocity);
             num("Miqp::UseBoxAsEnv", q.use_box_as_env); num("Miqp::WriteDebugFiles", q.write_debug_files);
             num("Miqp::DebugFilePath", q.debug_file_path); num("Miqp::DebugFilePrefix", q.debug_file_prefix);
             num("Miqp::MultiAgentPlanning", q.multi_agent_planning); num("Miqp::ObstaclesSoft", q.obstacles_soft);
             num("Miqp::PredictionErrorTimePercentage", q.prediction_error_time_percentage);
             return new BehaviorMiqpAgent(s, q);
           }),
           py::arg("params") = py::dict())
      .def("Plan",
           [agent_from](BehaviorMiqpAgent &b, double delta_time, const py::dict &world) {
             ObservedWorldLite w;
             w.time = world["time"].cast<double>();
             w.ego = agent_from(world["ego"].cast<py::dict>());
             if (world.contains("others")) for (auto h : world["others"].cast<py::list>()) w.others.push_back(agent_from(h.cast<py::dict>()));
             w.road_polygon = to_matrix(world["road_polygon"].cast<py::array_t<double, py::array::c_style | py::array::forcecast>>());
             const BehaviorMiqpAgent::Trajectory tr = b.Plan(delta_time, w);
             py::array_t<double> out({(py::ssize_t)tr.size(), (py::ssize_t)5});
             auto o = out.mutable_unchecked<2>();
             for (size_t k = 0; k < tr.size(); ++k) for (int c = 0; c < 5; ++c) o((py::ssize_t)k, c) = tr[k][c];
             return out;
           },
           py::arg("delta_time"), py::arg("observed_world"),
           "one planning cycle; observed_world = {time, ego: {id, state [x, y, theta, v, a], length, width, lane_center (n, 2)}, others: [...], road_polygon (k, 2)}; "
           "returns rows {t, x, y, theta, v}")
      .def_property_readonly("last_planning_success", &BehaviorMiqpAgent::GetLastPlanningSuccess)
      .def_property_readonly("last_solution_time", &BehaviorMiqpAgent::GetLastSolutionTime)
      .def_property_readonly("last_action", &BehaviorMiqpAgent::GetLastAction)
      .def_property_readonly("behavior_status", &BehaviorMiqpAgent::GetBehaviorStatus)
      .def_property_readonly("car_idxs", &BehaviorMiqpAgent::GetCarIdxs)
      .def_property_readonly("obstacle_ids", &BehaviorMiqpAgent::GetObstacleIds)
      .def_property_readonly("env_polygon", [](const BehaviorMiqpAgent &b) { return to_array(b.GetEnvironmentPolygon()); })
      .def("SetWarmstartType", &BehaviorMiqpAgent::SetWarmstartType)
      .def("GetLastSolutionProperties", [](BehaviorMiqpAgent &b) { return b.GetPlanner().GetSolutionProperties(); });

  py::enum_<OptimizationStatus>(m, "OptimizationStatus", py::arithmetic())
      .value("SUCCESS", OptimizationStatus::SUCCESS)
      .value("FAILED_NO_SOLUT", OptimizationStatus::FAILED_NO_SOLUT)
      .value("FAILED_SEG_FAULT", OptimizationStatus::FAILED_SEG_FAULT)
      .value("FAILED_TIMEOUT", OptimizationStatus::FAILED_TIMEOUT)
      .export_values();

  py::class_<SolutionProperties>(m, "SolutionProperties")
      .def(py::init())
      .def_readwrite("objective", &SolutionProperties::objective)
      .def_readwrite("status", &SolutionProperties::status)
      .def_readwrite("gap", &SolutionProperties::gap)
      .def_readwrite("time", &SolutionProperties::time)
      .def_readwrite("NrSolutionPool", &SolutionProperties::NrSolutionPool);

  py::enum_<MiqpPlannerWarmstartType>(m, "WarmstartType")
      .value("NO_WARMSTART", NO_WARMSTART)
      .value("RECEDING_HORIZON_WARMSTART", RECEDING_HORIZON_WARMSTART)
      .value("LAST_SOLUTION_WARMSTART", LAST_SOLUTION_WARMSTART)
      .value("BOTH_WARMSTART_STRATEGIES", BOTH_WARMSTART_STRATEGIES)
      .export_values();

  py::enum_<MiqpPlannerParallelMode>(m, "ParallelMode")
      .value("AUTO", AUTO)
      .value("DETERMINISTIC", DETERMINISTIC)
      .value("OPPORTUNISTIC", OPPORTUNISTIC)
      .export_values();
}
