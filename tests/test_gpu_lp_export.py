"""The CPLEX LP export of the C++ solver class (B200Wrapper::exportModel, what cplex.exportModel does in the reference,
src/cplex_wrapper.cpp:151-154) for cplexmodel_testcase.dat: the rows come from the device assembly kernel; the file is
parsed here and compared with the reference's pinned statistics (test/cplex_wrapper_test.cc:866-871) and, row by row,
with the oracle's instantiation of the same model."""
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu


def parse_lp(path):
    txt = open(path).read()
    body = txt.split("Subject To", 1)[1]
    cons, rest = body.split("Bounds", 1)
    bounds, bins = rest.split("Binaries", 1)
    rows = []
    for m in re.finditer(r"^ c(\d+):(.*?)(<=|>=|=)\s*(\S+)\s*$", cons.replace("\n     ", " "), flags=re.M):
        terms = re.findall(r"([+-])\s*([0-9.eE+-]+)\s+([A-Za-z_][^\s]*)", m.group(2))
        rows.append((int(m.group(1)), [(float(v) * (1 if sg == "+" else -1), name) for sg, v, name in terms], m.group(3), float(m.group(4))))
    binaries = bins.split("End")[0].split()
    free = re.findall(r"^ (\S+) free$", bounds, flags=re.M)
    boxed = re.findall(r"^ 0 <= (\S+) <= (\S+)$", bounds, flags=re.M)
    return rows, binaries, free, boxed, txt


def test_lp_export_matches_the_pinned_statistics_and_the_oracle_rows(testcase_problem, tmp_path):
    from test_host_api_cpp import _build, EXE, ROOT   # the C++ test writes the file
    _build()
    r = subprocess.run([EXE, "gpu", os.path.abspath(ROOT), str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    rows, binaries, free, boxed, txt = parse_lp(str(tmp_path / "miqp_b200_hostapi_testcase.lp"))
    p = testcase_problem
    # reference pins: 12361 rows, 29834 non-zeros, 1240 binaries, 340 continuous
    assert len(rows) == 12361
    assert sum(1 for _, t, _, _ in rows for c, n in t if n != "objconst") == 29834
    assert len(binaries) == 1240 and len(set(binaries)) == 1240
    assert len(free) + len(boxed) == 340
    assert all(hi == "1" for _, hi in boxed)                 # slackvarsObstacle in [0, 1]
    # row by row against the oracle (OPL order, exact-zero coefficients dropped)
    rowptr, cols, vals, lo, hi = O.build_rows(p)
    lay = O.layout(p)
    names = {}
    v = O.block_views(p, np.arange(lay.ncols, dtype=np.float64))
    for fam, arr in v.items():
        for idx in np.ndindex(arr.shape):
            names[int(arr[idx])] = fam + "".join(f"({k + 1})" for k in idx)
    for r_idx, terms, op, rhs in rows[::37] + rows[-5:]:
        k = r_idx - 1
        ref = {names[int(c)]: float(a) for c, a in zip(cols[rowptr[k]:rowptr[k + 1]], vals[rowptr[k]:rowptr[k + 1]]) if a != 0.0}
        got = {n: c for c, n in terms if n != "objconst"}
        assert set(got) == set(ref), (r_idx, got, ref)
        for n in ref:
            # the C++ ModelParameters keep the scalars as float like the reference's (ts = 0.2f), the oracle reads 0.2 from the file
            assert got[n] == pytest.approx(ref[n], rel=1e-7, abs=1e-300), (r_idx, n)
        if op == "=":
            assert lo[k] == hi[k] == pytest.approx(rhs, rel=1e-7, abs=1e-9)
        elif op == "<=":
            assert np.isinf(lo[k]) and hi[k] == pytest.approx(rhs, rel=1e-7, abs=1e-9)
        else:
            assert np.isinf(hi[k]) and lo[k] == pytest.approx(rhs, rel=1e-7, abs=1e-9)
    # objective: quadratic diagonal 2 w inside [ ] / 2 and the constant on objconst
    assert "objconst = 1" in txt and " ] / 2" in txt
    assert re.search(r"\+ 2 pos_x\(1\)\(1\) \^2", txt)        # WEIGHTS_POS_X = 1 in the fixture
