"""The planner-level solution pool (include/miqp_planner_solution_pool.h) is exported by libmiqp_planner_c_api.so and bound
by planner_capi; the C ABI of the solver library declares its pool entry points."""
import os
import re

from planner_miqp_b200 import planner_capi as PC
import planner_miqp_b200 as P

INCLUDE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")


def test_every_function_of_the_pool_header_is_exported():
    hdr = open(os.path.join(INCLUDE, "miqp_planner_solution_pool.h")).read()
    declared = re.findall(r"^\w[\w\s\*]*?\b(\w+CMiqpPlanner)\(", hdr, flags=re.M)
    assert sorted(declared) == sorted(PC.SOLUTION_POOL_SYMBOLS)
    lib = PC.load_library()
    assert all(hasattr(lib, s) for s in declared)


def test_solver_pool_entry_points_are_declared():
    hdr = open(os.path.join(INCLUDE, "miqp_b200.h")).read()
    for s in ("miqp_b200_set_solution_pool", "miqp_b200_pool_sizes", "miqp_b200_pool_fetch"):
        assert s in P.DECLARED_SYMBOLS and s + "(" in hdr
