// b200_wrapper.hpp -- host driver of the CUDA MIQP backend, shaped like the reference's
// solver class.
//
// Takes the place of CplexWrapper (reference src/cplex_wrapper.hpp:61-275): same method names,
// argument meaning and status / error convention, so MiqpPlanner and reference-side callers
// keep their code (`using CplexWrapper = B200Wrapper` below).  What callCplex() did through
// OPL + CPLEX (src/cplex_wrapper.cpp:65-249) is one call into libmiqp_b200.so:
//
//   ModelInputDataSource::read (src/model_input_data_source.cpp:180-275)  -> Flatten(): row-major
//       arrays, every real rounded to precision-2 decimals, polygons as closed edge lists
//   opl.generate() + cplex.solve() (:98, :158-185)                         -> miqp_b200_solve_batch
//   initializeWarmstart (:494-639)                                         -> MIP start vector
//   collectRawResults (:311-448), collectSolutionStatus (:672-678)         -> Unpack()
//   collectCplexStatistics (:680-690)                                      -> miqp_b200_sizes (opt-in)
//   printExternalData / solution dumps (:141-155, :212-229)                -> WriteParametersDat / WriteSolution
//
// There is no CPU fallback: without a usable CUDA device callCplex() returns FAILED_SEG_FAULT
// (the reference's status for "the solver could not run", src/cplex_wrapper.cpp:99-109) and
// lastError() says why.
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "../../include/miqp_b200.h"
#include "planner_data.hpp"

namespace miqp {
namespace planner {
namespace cplex {

// row-major copy of a ModelParameters that outlives the C struct pointing into it
struct FlatProblem {
  MiqpB200Problem p{};
  std::vector<std::vector<double>> d;
  std::vector<std::vector<int>> i;
};
// ModelParameters -> C ABI problem; reals rounded to `precision - 2` decimals (0 = no rounding)
void Flatten(const ModelParameters &m, int precision, FlatProblem &out);
// full column vector <-> RawResults (decision_variables.mod order, miqp_b200_layout)
void Unpack(const MiqpB200Layout &l, const double *x, RawResults &r);
void Pack(const MiqpB200Layout &l, const RawResults &r, bool relax_last_step, std::vector<double> &x);
// OPL .dat dialect of the reference's parameter dumps (readable by oracle/dat_io.py)
bool WriteParametersDat(const MiqpB200Problem &p, const ModelParameters &m, const std::string &path);
// names of the columns in decision_variables.mod order, OPL style with 1-based indices: pos_x(1)(2), active_region(1)(2)(32), ...
std::vector<std::string> ColumnNames(const MiqpB200Layout &l);
// CPLEX MIP-start file (.mst, XML) of a full column vector / back; what cplex.writeMIPStarts / readMIPStarts exchange
// (reference src/cplex_wrapper.cpp:128-138, 206-209)
bool WriteMst(const std::string &path, const MiqpB200Layout &l, const std::vector<double> &x);
bool ReadMst(const std::string &path, int ncols, std::vector<double> &x);

// member of the solution pool (miqp_b200_pool_fetch): objective and violation of its full column vector, device-evaluated
struct SolutionPoolEntry {
  double objective = 0.0, max_violation = 0.0;
  bool converged = false;   // the leaf QP was solved to optimality
  std::vector<double> x;    // full column vector (decision_variables.mod order): Unpack() gives its RawResults
};

class B200Wrapper {
 public:
  enum ParameterSource { DATFILE = 0, CPPINPUTS = 1, MIXED = 2 };
  typedef MiqpPlannerWarmstartType WarmstartType;

  B200Wrapper();
  explicit B200Wrapper(int precision);
  // modpath / modfile name the OPL model in the reference; accepted and ignored (the
  // formulation is compiled into the device kernels)
  B200Wrapper(const std::string &modpath, const std::string &modfile, ParameterSource source, int precision);
  B200Wrapper(const B200Wrapper &o);              // fresh device handle, results not copied
  B200Wrapper &operator=(const B200Wrapper &o);   // copies only the debug path
  ~B200Wrapper();

  void resetParameters(std::shared_ptr<ModelParameters> parameters) { parameters_ = parameters; }
  // copies only the solver options (time limit, gap, CPLEX emphasis switches) into the bound parameters
  // (reference src/cplex_wrapper.cpp:893, src/model_input_data_source.cpp:282-296)
  void overrideSolverSettingsDataSource(std::shared_ptr<ModelParameters> parameters);
  // DATFILE source: the OPL .dat file is read at every callCplex (host/dat_reader.hpp); values are taken as written
  void setParameterDatFileAbsolute(const char *datfile) { datFile_ = datfile; }
  void setParameterDatFileRelative(const char *datfile) { datFile_ = modPath_ + datfile; }
  void setParameterSource(ParameterSource src) { source_ = src; }
  void addRecedingHorizonWarmstart(std::shared_ptr<RawResults> warmstart, WarmstartType type);
  void setLastSolutionWarmstart(WarmstartType type);
  void deleteLastSolutionWarmstartFile();
  void setSpecialOrderedSets(bool in) { useSos_ = in; }
  void setUseBranchingPriorities(bool in) { useBranchingPriorities_ = in; }
  void setBranchingPriorityValueExtent(int start, int extent) { prioStart_ = start; prioExtent_ = extent; }
  void setBufferCplexOutputsToStream(bool in) { bufferOutputs_ = in; }
  void setDebugOutputPrint(bool in) { debugPrint_ = in; }
  void setDebugOutputFilePath(const std::string &path) { debugPath_ = path; }
  void setDebugOutputFilePrefix(const std::string &prefix) { debugPrefix_ = prefix; }
  std::string getDebugOutputParameterFilePath() const { return lastParameterFile_; }
  std::string getTmpWarmstartFile() const { return tmpWarmstartFile_; }
  void setTmpWarmstartFile(const std::string &path) { tmpWarmstartFile_ = path; }   // (the reference's path is fixed: src/cplex_wrapper.hpp:104)
  // CPLEX LP file of the big-M model of the bound parameters, rows instantiated on the device in OPL order
  // (cplex.exportModel, reference src/cplex_wrapper.cpp:151-154); exact-zero coefficients are dropped as CPLEX does
  bool exportModel(const std::string &lpfile);
  bool writeMIPStarts(const std::string &mstfile) const;   // last solution
  bool readMIPStarts(const std::string &mstfile);          // becomes the "last solution" MIP start
  void setCollectModelStatistics(bool in) { collectSizes_ = in; }   // rows / non-zeros cost one more device pass
  void setDevice(int ordinal);
  // Solution pool: up to `capacity` (0..64, 0 = off) best distinct feasible plans of every solve, entry 0 = the returned solution.
  // With the pool on, SolutionProperties.NrSolutionPool counts its entries.  Returns false for a capacity outside 0..64.
  bool setSolutionPoolCapacity(int capacity);
  int getSolutionPoolCapacity() const { return poolCapacity_; }
  const std::vector<SolutionPoolEntry> &getSolutionPool() const { return pool_; }
  // RawResults of pool entry j (false if there is no such entry)
  bool getSolutionPoolResults(int j, RawResults &out) const;

  // one MIQP solve of the bound ModelParameters; `timestamp` only names the debug files
  OptimizationStatus callCplex(double timestamp = 0.0);
  // the same for many independent problems in ONE device batch (multi-scenario dispatch)
  static std::vector<OptimizationStatus> callBatch(const std::vector<B200Wrapper *> &solvers, double timestamp = 0.0);
  // callBatch of the same solvers in the same order with receding-horizon warm starts: the previous incumbents are shifted on the
  // device instead of sending the host-side shifted vectors (on by default; off = always the host path of callCplex)
  void setDeviceWarmstart(bool on) { deviceWarmstart_ = on; }
  static long deviceWarmstartBatches() { return deviceWarmstartBatches_; }   // batches that took the device path so far

  std::shared_ptr<RawResults> getRawResults() const { return results_; }
  // injects a solution vector as if a solve had returned it (replay of recorded solutions, tests of the warm-start logic)
  bool setSolutionVector(const double *x, int ncols);
  SolutionProperties getSolutionProperties() const { return props_; }
  const std::vector<double> &getSolutionVector() const { return lastX_; }
  const std::string &lastError() const { return error_; }

 private:
  struct Prepared;
  bool Prepare(double timestamp, Prepared &out);
  OptimizationStatus Finish(const Prepared &pr, const MiqpB200SolveInfo &info, const double *x, double timestamp);
  bool EnsureSolver();
  bool FetchPool(MiqpB200Solver *solver, int k, const MiqpB200Layout &layout);

  std::shared_ptr<ModelParameters> parameters_;
  std::shared_ptr<RawResults> results_;
  SolutionProperties props_;
  int precision_ = 12;
  int device_ = 0;
  MiqpB200Solver *solver_ = nullptr;
  bool useSos_ = false, useBranchingPriorities_ = false, bufferOutputs_ = false, debugPrint_ = false, collectSizes_ = false;
  int prioStart_ = 1, prioExtent_ = 0;
  std::string debugPath_, debugPrefix_, lastParameterFile_, error_;
  ParameterSource source_ = CPPINPUTS;
  std::string modPath_, datFile_;
  std::string tmpWarmstartFile_ = "/tmp/warmstart_debug_res.mst";
  // MIP starts
  std::shared_ptr<RawResults> recedingWarm_;
  bool deviceWarmstart_ = true;
  std::vector<B200Wrapper *> lastBatch_;      // members of the last successful batch run on this solver's handle
  static long deviceWarmstartBatches_;
  bool useRecedingWarm_ = false, useLastSolution_ = false;
  std::vector<double> lastX_;           // last solution vector (the ".mst" of the reference)
  MiqpB200Layout lastLayout_{};
  bool haveLast_ = false;
  int poolCapacity_ = 0;
  std::vector<SolutionPoolEntry> pool_;   // of the last solve
  MiqpB200Layout poolLayout_{};
};

typedef B200Wrapper CplexWrapper;   // reference-side code keeps its spelling

}  // namespace cplex
}  // namespace planner
}  // namespace miqp
