// C++ API test of the host side (planner-miqp_b200/host): the class-level behaviour the reference's gtest
// suites check on MiqpPlanner / CplexWrapper (test/miqp_planner_test.cc, test/cplex_wrapper_test.cc) that needs
// no BARK.  `test_host_api cpu|gpu <repository root> <scratch directory>`: `cpu` runs the device-free part, `gpu` adds
// the solves.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>

#include "../../planner-miqp_b200/host/dat_reader.hpp"
#include "../../planner-miqp_b200/host/miqp_planner.hpp"

using namespace miqp::planner;
using miqp::planner::cplex::CplexWrapper;

static int failures = 0;
static std::string g_tmp;    // directory the test writes its files to (argv[3]; one per run, so runs of other users cannot collide)
#define CHECK(c) do { if (!(c)) { std::printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #c); ++failures; } } while (0)

static PolyLine Line(std::initializer_list<double> pts, double inc = 0.2) {
  std::vector<double> v(pts);
  return PolyLine(v.data(), (int)v.size() / 2, inc);
}

static void cpu_part() {
  Settings s = DefaultSettings();
  CHECK(s.nr_regions == 16 && s.nr_steps == 20 && s.precision == 12 && std::fabs(s.ts - 0.25f) < 1e-7);
  CHECK(std::string(ApolloDefaultSettings().cplexModelpath).find("cplex_modfiles") != std::string::npos);
  MiqpPlanner planner(s);
  auto p = planner.GetParameters();
  CHECK(p->nr_regions == 16 && p->NumSteps == 20 && p->NumCars == 0);
  CHECK(p->fraction_parameters.rows() == 16 && p->poly_orientation_params.POLY_SINT_UB.rows() == 16);
  // test/miqp_planner_test.cc:127-134 spot value of the 16-region sine table
  const double st[6] = {0, 4, 0, 0, 0.1, 0};
  int idx = planner.AddCar(st, Line({0, 0, 50, 0}), 5, 1);
  CHECK(idx == 0 && p->NumCars == 1);
  CHECK(p->IntitialState(0, MIQP_STATE_VX) == 4 && p->x_ref.cols() == 20);
  CHECK(std::fabs(p->WEIGHTS_POS_X(0) - 1.0) < 1e-12 && std::fabs(p->WEIGHTS_JERK_X(0) - 0.5) < 1e-12);   // lambda 0.5 * weight
  CHECK(p->possible_region(0, 0) == 1 && p->possible_region(0, 15) == 1 && p->possible_region(0, 1) == 1 && p->possible_region(0, 8) == 0);
  CHECK(std::fabs(p->total_max_acc - (float)(p->acc_limit_params.max_x.maxCoeff() + 1e-6)) < 1e-5 || p->total_max_acc >= p->acc_limit_params.max_y.maxCoeff());
  const double st2[6] = {0, 4, 0, 4, 0.1, 0};
  int idx2 = planner.AddCar(st2, Line({0, 4, 50, 4}), 5, 1, 0.0, false);
  CHECK(idx2 == 1 && p->NumCars == 2 && p->WEIGHTS_POS_X(1) == 0 && p->WEIGHTS_VEL_X(1) == 2);   // untracked positions
  int idx3 = planner.AddCar(st2, Line({0, 8, 50, 8}), 5, 1);
  CHECK(idx3 == 2);
  bool threw = false;
  try { planner.RemoveCar(1); } catch (const NotImplementedException &) { threw = true; }
  CHECK(threw);                                   // middle cars cannot be removed (src/miqp_planner.cpp:553-557)
  planner.RemoveCar(2);
  CHECK(p->NumCars == 2 && p->x_ref.rows() == 2);
  planner.RemoveCar(0);                            // ego: refused, logged
  CHECK(p->NumCars == 2);
  threw = false;
  try { planner.RemoveObstacle(0); } catch (const NotImplementedException &) { threw = true; }
  CHECK(threw);
  int oid = planner.AddObstacle({{20.0, 0.0, 0.0}}, 1.0, 1.0, false, true);
  CHECK(oid == 0 && p->nr_obstacles == 1 && p->max_lines_obstacles == 4 && (int)p->ObstacleConvexPolygon[0].size() == 20);
  CHECK(std::fabs(p->ObstacleConvexPolygon[0][0](0, 0) - 18.5) < 1e-12);   // 1 x 1 box inflated by the collision radius
  planner.RemoveAllObstacles();
  CHECK(p->nr_obstacles == 0 && p->max_lines_obstacles == 0);
  // copies share the parameters and get their own solver (src/miqp_planner.cpp:153-175)
  MiqpPlanner copy(planner);
  CHECK(copy.GetParameters().get() == p.get());
  CHECK(copy.GetCplexWrapper().getRawResults().get() != planner.GetCplexWrapper().getRawResults().get());
  {   // non-convex road polygons are decomposed (reference: ConvexifiedMap::Convert); a rejected map makes Plan() fail closed
    MiqpPlanner mp(s);
    const double lv[12] = {0, 0, 50, 0, 50, 10, 10, 10, 10, 40, 0, 40};
    MatrixXd L(6, 2);
    for (int k = 0; k < 6; ++k) { L(k, 0) = lv[2 * k]; L(k, 1) = lv[2 * k + 1]; }
    CHECK(mp.UpdateConvexifiedMap(L));
    const double s0[6] = {5, 4, 0, 5, 0.1, 0};
    mp.AddCar(s0, Line({5, 5, 45, 5}), 5, 1);
    MatrixXd degenerate(3, 2);
    for (int k = 0; k < 3; ++k) { degenerate(k, 0) = k; degenerate(k, 1) = 0; }
    CHECK(!mp.UpdateConvexifiedMap(degenerate));
    CHECK(!mp.Plan(0.0));                          // no environment, no plan
    CHECK(mp.UpdateConvexifiedMap(L));              // accepted again
  }
  // unknown table combination
  Settings bad = DefaultSettings(); bad.nr_regions = 64;
  threw = false;
  try { MiqpPlanner q(bad); } catch (const std::invalid_argument &) { threw = true; }
  CHECK(threw);
  // state conversions of the facade
  double ms[6];
  MiqpPlanner::CarStateToMiqpState(1.f, 2.f, (float)M_PI / 2, 3.f, 0.5f, ms);
  CHECK(ms[MIQP_STATE_X] == 1.0 && ms[MIQP_STATE_Y] == 2.0 && std::fabs(ms[MIQP_STATE_VX]) < 1e-6 && std::fabs(ms[MIQP_STATE_VY] - 3.0) < 1e-6 && std::fabs(ms[MIQP_STATE_AY] - 0.5) < 1e-6);
  CHECK(MiqpPlanner::IsVxVyValid(0.71, 0.0) && MiqpPlanner::IsVxVyValid(0.0, -0.8) && !MiqpPlanner::IsVxVyValid(0.7, -0.7));
  // the solver class keeps the reference's configuration surface
  CplexWrapper w("cplexmodel/", "cplexmodel.mod", CplexWrapper::CPPINPUTS, 12);
  w.setSpecialOrderedSets(true); w.setUseBranchingPriorities(true); w.setBranchingPriorityValueExtent(1, 19);
  w.setBufferCplexOutputsToStream(true); w.setDebugOutputPrint(false);
  CHECK(w.getTmpWarmstartFile() == "/tmp/warmstart_debug_res.mst");
  CHECK(w.callCplex(0.0) == FAILED_SEG_FAULT);     // no parameters bound: the solver cannot run
  // flatten / pack / unpack round trip
  miqp::planner::cplex::FlatProblem f;
  miqp::planner::cplex::Flatten(*p, 12, f);
  MiqpB200Layout l;
  CHECK(miqp_b200_layout(&f.p, &l) == MIQP_B200_OK);
  CHECK(l.ncols == 12 * 2 * 20 + 2 * 20 * 16 + 5 * 2 * 20 + 16 * 20 + 4 * 20);
  std::vector<double> x(l.ncols);
  for (int k = 0; k < l.ncols; ++k) x[k] = (k < l.base_nwe) ? 0.25 * k : (double)(k % 2);
  RawResults r; std::vector<double> y;
  miqp::planner::cplex::Unpack(l, x.data(), r);
  miqp::planner::cplex::Pack(l, r, false, y);
  bool same = true;
  for (int k = 0; k < l.ncols; ++k) same = same && (k >= l.base_sv ? y[k] == (double)(int)x[k] : y[k] == x[k]);
  CHECK(same);
  miqp::planner::cplex::Pack(l, r, true, y);
  CHECK(std::isnan(y[l.base_ar + 19 * 16]) && !std::isnan(y[l.base_ar + 18 * 16]) && !std::isnan(y[19]));
  // column names in OPL style, .mst round trip (cplex.writeMIPStarts / readMIPStarts, src/cplex_wrapper.cpp:128-138, 206-209)
  const std::vector<std::string> names = miqp::planner::cplex::ColumnNames(l);
  CHECK((int)names.size() == l.ncols && names[0] == "u_x(1)(1)" && names[2 * 2 * 20 + 20 + 3] == "pos_x(2)(4)");
  CHECK(names[l.base_ar + (1 * 20 + 2) * 16 + 5] == "active_region(2)(3)(6)" && names[l.base_rcna + 4 * 2 * 20] == "region_change_not_allowed_combined(1)(1)");
  CHECK(names[l.base_c2c + 17] == "car2car_collision(1)(1)(2)(2)" && names[l.ncols - 1] == "slackvars(1)(1)(20)(4)");
  const std::string mst = g_tmp + "/miqp_b200_test_roundtrip.mst";
  CHECK(miqp::planner::cplex::WriteMst(mst, l, x));
  std::vector<double> xr;
  CHECK(miqp::planner::cplex::ReadMst(mst, l.ncols, xr) && xr == x);
  CHECK(!miqp::planner::cplex::ReadMst(mst, l.ncols - 1, xr) && !miqp::planner::cplex::ReadMst("/nonexistent.mst", l.ncols, xr));
  {   // a wrapper bound to the same parameters takes the file as its "last solution" MIP start and writes it back unchanged
    CplexWrapper w2(12);
    w2.resetParameters(p);
    CHECK(!w2.writeMIPStarts(g_tmp + "/miqp_b200_test_none.mst"));      // nothing solved or read yet
    CHECK(w2.readMIPStarts(mst) && w2.getSolutionVector() == x);
    CHECK(w2.writeMIPStarts(g_tmp + "/miqp_b200_test_roundtrip2.mst") && miqp::planner::cplex::ReadMst(g_tmp + "/miqp_b200_test_roundtrip2.mst", l.ncols, xr) && xr == x);
    w2.setTmpWarmstartFile(g_tmp + "/miqp_b200_test_tmpws.mst");
    CHECK(w2.getTmpWarmstartFile() == g_tmp + "/miqp_b200_test_tmpws.mst");
    // overrideSolverSettingsDataSource copies the solver options only (src/model_input_data_source.cpp:282-296)
    auto o = std::make_shared<ModelParameters>();
    o->max_solution_time = 3.5f; o->relative_mip_gap_tolerance = 0.02f; o->mipemphasis = 1; o->parallelmode = -1; o->NumSteps = 7;
    const int steps = p->NumSteps;
    w2.overrideSolverSettingsDataSource(o);
    CHECK(p->max_solution_time == 3.5f && p->relative_mip_gap_tolerance == 0.02f && p->mipemphasis == 1 && p->parallelmode == -1 && p->NumSteps == steps);
  }
}

static std::string g_root;   // repository root (argv[2])

// .dat dialect: the reference fixture parses into ModelParameters, and a written dump reads back unchanged
static void dat_part() {
  ModelParameters m;
  datio::ReadParametersDat(g_root + "/tests/golden/cplexmodel_testcase.dat", m);
  CHECK(m.NumSteps == 20 && m.nr_regions == 32 && m.NumCars == 1 && m.nr_obstacles == 1 && m.nr_environments == 1 && m.max_lines_obstacles == 4);
  CHECK(std::fabs(m.ts - 0.2f) < 1e-7 && std::fabs(m.relative_mip_gap_tolerance - 0.1f) < 1e-7 && m.max_solution_time == 60.f);
  CHECK(m.IntitialState(0, MIQP_STATE_VX) == 5.0 && m.IntitialState(0, MIQP_STATE_VY) == 0.1 && m.x_ref(0, 19) == 19.0);
  CHECK(m.ObstacleConvexPolygon.size() == 1 && m.ObstacleConvexPolygon[0].size() == 20 && m.ObstacleConvexPolygon[0][0].rows() == 4);
  CHECK(m.ObstacleConvexPolygon[0][3](0, 0) == 23.0 && m.ObstacleConvexPolygon[0][3](0, 1) == -1.0 && m.ObstacleConvexPolygon[0][3](2, 0) == 17.0);
  CHECK(m.fraction_parameters.rows() == 32 && m.poly_curvature_params.POLY_KAPPA_AX_MAX.rows() == 32 && m.obstacle_is_soft[0] == 0);
  cplex::FlatProblem f1, f2;
  cplex::Flatten(m, 0, f1);
  const std::string tmp = g_tmp + "/miqp_b200_test_roundtrip.dat";
  CHECK(cplex::WriteParametersDat(f1.p, m, tmp));
  ModelParameters m2;
  datio::ReadParametersDat(tmp, m2);
  cplex::Flatten(m2, 0, f2);
  CHECK(f1.p.N == f2.p.N && f1.p.R == f2.p.R && f1.p.O == f2.p.O && f1.p.E == f2.p.E && f1.p.ts == f2.p.ts);
  bool same = f1.d.size() == f2.d.size();
  for (size_t k = 0; same && k < f1.d.size(); ++k) same = (f1.d[k] == f2.d[k]);   // 12 printed digits reproduce every fixture value
  CHECK(same);
  bool threw = false;
  try { datio::ReadParametersDat("/nonexistent.dat", m2); } catch (const std::runtime_error &) { threw = true; }
  CHECK(threw);
}

static void gpu_part() {
  Settings s = DefaultSettings();
  s.relative_mip_gap_tolerance = 1e-4f;
  s.warmstartType = RECEDING_HORIZON_WARMSTART;
  MatrixXd map(4, 2);
  const double mv[8] = {-50, -50, -50, 50, 50, 50, 50, -50};
  for (int k = 0; k < 4; ++k) { map(k, 0) = mv[2 * k]; map(k, 1) = mv[2 * k + 1]; }
  MiqpPlanner planner(s, map);
  double st[6] = {0, 4, 0, 0, 0.1, 0};
  const PolyLine ref = Line({0, 0, 50, 0});
  planner.AddCar(st, ref, 5, 1);
  planner.GetCplexWrapper().setCollectModelStatistics(true);
  CHECK(planner.Plan(0.0));
  auto p = planner.GetParameters();
  CHECK(p->initial_region(0) == 1 && p->nr_environments == 1 && (int)p->MultiEnvironmentConvexPolygon.size() == 1);
  SolutionProperties sp = planner.GetSolutionProperties();
  CHECK(sp.status == 101 || sp.status == 102);
  CHECK(sp.gap <= 1e-4 && sp.max_violation <= 1e-6 && sp.NrSolutionPool == 1);
  CHECK(sp.NrBinaryVariables == 5 * 20 + 16 * 20 + 5 * 20);
  CHECK(sp.NrFloatVariables == 240);
  // rows depend on the number of possible regions (3 here); test_sos.dat with all 16 possible has 8944
  CHECK(sp.NrConstraints > 5000 && sp.NrConstraints < 8944 && sp.NonZeroCoefficients > sp.NrConstraints);
  auto rr = planner.GetSolution();
  CHECK(rr->N == 20 && rr->NrCars == 1 && rr->pos_x(0, 0) == 0.0 && rr->active_region(0, 0, 0) == 1);
  for (int i = 0; i < 20; ++i) { int sum = 0; for (int j = 0; j < 16; ++j) sum += rr->active_region(0, i, j); CHECK(sum == 1); }
  CHECK(planner.HasValidWarmstart());
  {   // {t, x, y, theta, v} rows of the plan; the car drives along +x at about 4-5 m/s
    const std::vector<std::array<double, 5>> tr = planner.GetTrajectory(0, 1.0);
    CHECK(tr.size() == 20 && tr[0][0] == 1.0 && std::fabs(tr[1][0] - 1.25) < 1e-12 && tr[0][1] == 0.0);
    CHECK(std::fabs(tr[0][3] - std::atan2(0.1, 4.0)) < 1e-9 && std::fabs(tr[0][4] - std::sqrt(16.01)) < 1e-9 && tr[19][1] > 15.0);
  }
  // receding horizon: the next plan starts from the shifted solution and reaches the same objective as a cold planner
  double nxt[6]; planner.Get2ndOrderStateFromSolution(1, 0, nxt);
  planner.UpdateCar(0, nxt, ref);
  CHECK(planner.Plan(0.25));
  Settings sc = s; sc.warmstartType = NO_WARMSTART;
  MiqpPlanner cold(sc, map);
  cold.AddCar(nxt, ref, 5, 1);
  CHECK(cold.Plan(0.25));
  const double a = planner.GetSolutionProperties().objective, b = cold.GetSolutionProperties().objective;
  CHECK(std::fabs(a - b) <= 2e-4 * std::fabs(b));
  // infeasible start: obstacle on top of the car -> FAILED_NO_SOLUT for every region combination -> Plan() false
  MiqpPlanner blocked(sc, map);
  blocked.AddCar(st, ref, 5, 1);
  CHECK(blocked.AddObstacle({{0.0, 0.0, 0.0}}, 4.0, 4.0, false, true) == 0);
  CHECK(!blocked.Plan(0.0));
  SolutionProperties bp = blocked.GetSolutionProperties();
  CHECK(std::isnan(bp.objective) && std::isnan(bp.gap) && bp.status == 103);
  // DATFILE source (reference test/cplex_wrapper_test.cc:474-505): the dump written by a CPPINPUTS solve, solved again
  // from the file, gives the same objective and gap
  {
    MiqpPlanner src(sc, map);
    src.AddCar(st, ref, 5, 1);
    src.AddObstacle({{20.0, 1.0, 0.0}}, 2.0, 1.0, false, true);
    src.ActivateDebugFileWrite(g_tmp, "miqp_b200_hostapi_");
    CHECK(src.Plan(7.0));
    const std::string dump = src.GetCplexWrapper().getDebugOutputParameterFilePath();
    CHECK(!dump.empty());
    CplexWrapper fromfile("", "cplexmodel.mod", CplexWrapper::DATFILE, 12);
    fromfile.setParameterDatFileAbsolute(dump.c_str());
    CHECK(fromfile.callCplex(7.0) == SUCCESS);
    const SolutionProperties a1 = src.GetSolutionProperties(), a2 = fromfile.getSolutionProperties();
    CHECK(std::fabs(a1.objective - a2.objective) <= 1e-7 * std::fabs(a1.objective) && a2.gap <= 1e-4);
    // the reference fixture through the same path: known optimum 9.57603 (test/cplex_wrapper_test.cc:874)
    CplexWrapper fixture("", "cplexmodel.mod", CplexWrapper::DATFILE, 12);
    fixture.setParameterDatFileAbsolute((g_root + "/tests/golden/cplexmodel_testcase.dat").c_str());
    CHECK(fixture.callCplex(0.0) == SUCCESS);
    CHECK(std::fabs(fixture.getSolutionProperties().objective - 9.57603) <= 0.1 * 9.57603);   // the file asks for a 10 % gap
  }
  // .lp export of the reference fixture (cplex.exportModel, src/cplex_wrapper.cpp:151-154): the device-instantiated rows as a
  // CPLEX LP file; tests/test_gpu_lp_export.py parses it and compares it with the oracle's rows
  {
    CplexWrapper fx("", "cplexmodel.mod", CplexWrapper::DATFILE, 12);
    fx.setParameterDatFileAbsolute((g_root + "/tests/golden/cplexmodel_testcase.dat").c_str());
    fx.setLastSolutionWarmstart(LAST_SOLUTION_WARMSTART);
    fx.setTmpWarmstartFile(g_tmp + "/miqp_b200_hostapi_ws.mst");
    fx.deleteLastSolutionWarmstartFile();
    CHECK(fx.callCplex(0.0) == SUCCESS);
    CHECK(fx.exportModel(g_tmp + "/miqp_b200_hostapi_testcase.lp"));
    // LAST_SOLUTION_WARMSTART wrote the solution to the warm-start file; a fresh wrapper starts from it
    std::vector<double> xr;
    CHECK(miqp::planner::cplex::ReadMst(g_tmp + "/miqp_b200_hostapi_ws.mst", (int)fx.getSolutionVector().size(), xr) && xr == fx.getSolutionVector());
    CplexWrapper fy("", "cplexmodel.mod", CplexWrapper::DATFILE, 12);
    fy.setParameterDatFileAbsolute((g_root + "/tests/golden/cplexmodel_testcase.dat").c_str());
    fy.setLastSolutionWarmstart(LAST_SOLUTION_WARMSTART);
    fy.setTmpWarmstartFile(g_tmp + "/miqp_b200_hostapi_ws.mst");
    CHECK(fy.callCplex(1.0) == SUCCESS);
    CHECK(std::fabs(fy.getSolutionProperties().objective - fx.getSolutionProperties().objective) <= 0.1 * 9.57603);
    CHECK(fy.getSolutionProperties().NrNodes <= fx.getSolutionProperties().NrNodes);   // the MIP start is an incumbent from the first round on
  }
  // batched dispatch
  MiqpPlanner p1(sc, map), p2(sc, map);
  double s1[6] = {0, 3, 0, 0.5, 0.1, 0}, s2[6] = {0, 6, 0, -0.5, 0.1, 0};
  p1.AddCar(s1, ref, 5, 1); p2.AddCar(s2, ref, 5, 1);
  std::vector<bool> ok = MiqpPlanner::PlanBatch({&p1, &p2, &blocked}, 0.0);
  CHECK(ok.size() == 3 && ok[0] && ok[1] && !ok[2]);
}

int main(int argc, char **argv) {
  g_root = (argc > 2) ? argv[2] : ".";
  g_tmp = (argc > 3) ? argv[3] : "/tmp";
  cpu_part();
  dat_part();
  if (argc > 1 && std::strcmp(argv[1], "gpu") == 0) gpu_part();
  std::printf(failures ? "%d check(s) failed\n" : "all checks passed\n", failures);
  return failures ? 1 : 0;
}
