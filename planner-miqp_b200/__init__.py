"""planner-miqp_b200: B200-native MIQP backend for the planner-miqp motion-planning model.

The product is ``libmiqp_b200.so`` (hand-written sm_100a CUDA behind the C ABI of
``include/miqp_b200.h``); this package is the thin host-side binding.  There is no CPU
fallback: solving without a CUDA device raises.
"""
from .capi import (MiqpB200Error, Solver, PipelinedSolver, SolveInfo, Incumbent, library_path, load_library,  # noqa: F401
                   exported_symbols, DECLARED_SYMBOLS)
