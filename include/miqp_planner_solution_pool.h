/*
 * miqp_planner_solution_pool.h -- solution pool of the planner-level C ABI (libmiqp_planner_c_api.so).
 *
 * Beside the plan PlanCMiqpPlanner / PlanBatchCMiqpPlanner return, a planner can keep up to `capacity` further distinct
 * feasible plans the device search solved on the way (CPLEX's solution pool; its size is SolutionProperties.NrSolutionPool),
 * best first: the next-best manoeuvre when a downstream check rejects the first one, or the cost of passing an obstacle on the
 * other side.  Entry 0 is the plan GetRawCMiqpTrajectoryCMiqpPlanner returns.  Kept apart from miqp_planner_c_api.h, whose
 * entry points mirror the reference's library.
 */
#ifndef MIQP_PLANNER_SOLUTION_POOL_HEADER
#define MIQP_PLANNER_SOLUTION_POOL_HEADER

#include "miqp_planner_c_api.h"

#ifdef __cplusplus
extern "C" {
#endif

/* capacity 0..64 (0 = off, the default); applies from the next Plan().  Returns false for a capacity outside 0..64. */
bool SetSolutionPoolCapacityCMiqpPlanner(CMiqpPlanner c_miqp_planner, int capacity);
/* entries of the last Plan() (0 if the pool is off or the plan failed) */
int GetSolutionPoolSizeCMiqpPlanner(CMiqpPlanner c_miqp_planner);
/* trajectory of car carIdx in entry j, filled like GetRawCMiqpTrajectoryCMiqpPlanner; returns the entry's objective
 * (NaN and size 0 if there is no entry j) */
double GetSolutionPoolTrajectoryCMiqpPlanner(CMiqpPlanner c_miqp_planner, int j, int carIdx, double start_time,
                                             double *trajectory, MIQP_SIZE_OUT size);

#ifdef __cplusplus
}
#endif
#endif /* MIQP_PLANNER_SOLUTION_POOL_HEADER */
