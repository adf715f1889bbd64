"""Incumbent deliveries of frontier sharding without a device: the C ABI declares, exports and lists the export / merge entry
points, the ctypes mirror of the callback type matches the header, no source names a batched copy, and the node kernels keep
their ptxas figures while the new summary and merge kernels do not spill."""
import ctypes as C
import os
import re

import planner_miqp_b200 as P
from planner_miqp_b200 import capi
from test_anytime_symbols import BATCHED_COPIES, ptxas_figures

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENTRY_POINTS = ("miqp_b200_frontier_inc_export", "miqp_b200_frontier_inc_merge")


def header():
    return open(os.path.join(ROOT, "include", "miqp_b200.h")).read()


def test_entry_points_are_declared_exported_and_listed():
    hdr = header()
    table = hdr[:hdr.index("*/")]            # the table of entry points at the top of the header
    assert "miqp_b200_frontier_inc_export" in table and "_frontier_inc_merge" in table
    for name in ENTRY_POINTS:
        assert re.search(r"\bint " + name + r"\(", hdr), name
        assert name in P.DECLARED_SYMBOLS
        assert hasattr(P.load_library(), name)


def test_callback_type_mirrors_the_header():
    hdr = header()
    assert ("typedef int (*MiqpB200FrontierIncumbentFound)(void *user, int k, int rank, const double *traj, "
            "const MiqpB200Incumbent *inc);") in hdr
    f = capi.FRONTIER_INCUMBENT_FOUND
    assert f._restype_ is C.c_int
    assert list(f._argtypes_) == [C.c_void_p, C.c_int, C.c_int, capi._dp, C.POINTER(capi.CIncumbent)]
    lib = P.load_library()
    assert lib.miqp_b200_frontier_inc_merge.argtypes[4] is f
    # Incumbent gains a trailing rank; the positional construction of run_anytime stays valid
    inc = P.Incumbent(1.0, 0.0, 1.0, 0.5, 0.5, 0.1, 3, 10, 20, 7)
    assert inc.rank == -1 and P.Incumbent(*([0.0] * 6 + [0] * 4), 1).rank == 1


def test_no_source_names_a_batched_copy():
    hits = []
    for top in ("planner-miqp_b200", "tools", "tests", "include", "oracle", "."):
        for dirpath, dirs, files in os.walk(os.path.join(ROOT, top)):
            if top == ".":
                dirs[:] = []                # only the files at the root
            dirs[:] = [d for d in dirs if not d.startswith(".") and d != "__pycache__"]
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h", ".c", ".sh")):
                    text = open(os.path.join(dirpath, f), errors="replace").read()
                    hits += [(os.path.join(dirpath, f), n) for n in BATCHED_COPIES if n in text]
    assert hits == []


def test_node_kernels_keep_their_figures_and_the_new_kernels_do_not_spill(tmp_path):
    figs = ptxas_figures(["bnb.cu", "bnb_multi.cu"], tmp_path)
    for nw in (2, 4, 8):
        f = next(v for k, v in figs.items() if "bnb_nodes_kernelILi%dE" % nw in k)
        assert f["regs"] == 255 and f["stack"] == 480 and 164 <= f["spill"] <= 212, (nw, f)
    f = next(v for k, v in figs.items() if "bnb_nodes_multi_kernel" in k)
    assert f["regs"] == 249 and f["spill"] == 0, f
    new = {k: v for k, v in figs.items() if "bnb_frontier_inc_" in k and "_kernel" in k}
    assert len(new) == 3, sorted(new)
    assert all(v["spill"] == 0 and v["stack"] == 0 for v in new.values()), new
