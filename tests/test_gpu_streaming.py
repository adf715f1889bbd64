"""Streaming runs (miqp_b200_batch_run_streaming / Solver.run_streaming): every plan is handed to the caller once, in the round
its search ends, with the result batch_fetch_compact gives for it after the run; the run computes what batch_run computes.
The batches mix single-car plans (warp-team node kernel) and two-car plans (CTA-per-node kernel)."""
import copy
import ctypes as C

import numpy as np
import pytest

import planner_miqp_b200 as P
from planner_miqp_b200 import capi
from planner_miqp_b200.scenarios import obstacle_scenario, parallel_lanes, two_agent_merge, advance_obstacle_scenario

pytestmark = pytest.mark.gpu

GAP = 1e-4
NPLANS = 256
INFO_FIELDS = ("status", "proven", "objective", "best_bound", "gap", "seconds", "max_violation", "nodes", "qp_iters", "rounds",
               "uncertified", "pool_exhausted")


@pytest.fixture(scope="module")
def batch(testcase_problem):
    return ([obstacle_scenario(k).build() for k in range(NPLANS)] + [testcase_problem]
            + [parallel_lanes(2, nr_steps=5).build(), two_agent_merge(0, nr_steps=8).build(), two_agent_merge(1, nr_steps=8).build()])


def same(a, b):
    """bit-identical values (NaN included)"""
    if isinstance(a, float) or isinstance(b, float):
        return np.float64(a).tobytes() == np.float64(b).tobytes()
    return a == b


def assert_info(a, b, skip=("rounds",)):
    for f in INFO_FIELDS:
        if f not in skip:
            assert same(getattr(a, f), getattr(b, f)), (f, getattr(a, f), getattr(b, f))


def stream(s):
    got = []
    ms = s.run_streaming(lambda k, t, i: got.append((k, t, i)))
    assert ms > 0
    return got


def check_delivery(got, n, tr, infos, final_rounds):
    """each plan once, equal to the compact fetch after the run; rounds never decrease, k ascends within a round"""
    assert sorted(k for k, _, _ in got) == list(range(n))
    for k, t, i in got:
        assert np.array_equal(t, tr[k]), k
        assert_info(i, infos[k])
        assert i.rounds <= final_rounds
    rounds = [i.rounds for _, _, i in got]
    assert all(a <= b for a, b in zip(rounds, rounds[1:])), rounds
    for (ka, _, ia), (kb, _, ib) in zip(got, got[1:]):
        if ia.rounds == ib.rounds:
            assert ka < kb


@pytest.fixture(scope="module")
def streamed(batch):
    s = P.Solver()
    s.upload(batch, gap_tol=GAP, time_limit=60)
    got = stream(s)
    tr, infos = s.fetch_compact()
    xs, full = s.fetch()
    yield s, got, tr, infos, xs, full
    s.close()


def test_every_plan_once_equal_to_the_fetch_after_the_run(batch, streamed):
    s, got, tr, infos, xs, full = streamed
    final = s.run_stats()["rounds"]
    check_delivery(got, len(batch), tr, infos, final)
    for a, b in zip(infos, full):
        assert_info(a, b, skip=())
    # the same upload run by batch_run on a fresh solver: the same results
    s0 = P.Solver()
    s0.upload(batch, gap_tol=GAP, time_limit=60)
    s0.run()
    xs0, full0 = s0.fetch()
    tr0, _ = s0.fetch_compact()
    assert s0.run_stats()["rounds"] == final
    for k in range(len(batch)):
        assert np.array_equal(xs[k], xs0[k]), k
        assert np.array_equal(tr[k], tr0[k]), k
        assert_info(full[k], full0[k], skip=("seconds",))
    for k in (0, NPLANS, len(batch) - 1):
        assert np.array_equal(s.fetch_vector(k), s0.fetch_vector(k))
    assert s.run_stats()["nodes"] == s0.run_stats()["nodes"]
    s0.close()
    # a plain run after a streaming run on the same solver is a plain run again
    s.run()
    xs1, full1 = s.fetch()
    for k in range(len(batch)):
        assert np.array_equal(xs1[k], xs0[k])
        assert_info(full1[k], full0[k], skip=("seconds",))


def test_plans_arrive_before_the_batch_ends(batch, streamed):
    s, got, tr, infos, _, _ = streamed
    final = infos[0].rounds
    early = [k for k, _, i in got if i.rounds < final]
    assert len(early) >= len(batch) // 2, (len(early), final)
    assert got[0][2].rounds < final
    # every plan proven here finished in its search, so it arrived in the round select marked it finished
    for k, _, i in got:
        if i.proven:
            assert i.rounds < final
    print("plans delivered before the last round: %d of %d (%d rounds)" % (len(early), len(batch), final))


def test_time_limits_and_round_cap(batch):
    ps = batch[:48] + batch[NPLANS:]
    tiny = set(range(0, 48, 5))
    short = set(range(2, 48, 7)) - tiny
    lim = []
    for k, p in enumerate(ps):
        q = copy.copy(p)
        q.scal = dict(p.scal, max_solution_time=1e-9 if k in tiny else 2e-3 if k in short else 60.0)
        lim.append(q)
    s = P.Solver()
    s.upload(lim, gap_tol=GAP)
    got = stream(s)
    tr, infos = s.fetch_compact()
    check_delivery(got, len(ps), tr, infos, s.run_stats()["rounds"])
    for k in tiny:
        assert infos[k].status == 3 and not infos[k].proven      # FAILED_TIMEOUT: stopped before its first node
    # a round cap: the plans still searching when the batch stops are delivered once, at the end
    s = P.Solver(max_rounds=4)
    s.upload(ps, gap_tol=GAP, time_limit=60)
    got = stream(s)
    tr, infos = s.fetch_compact()
    final = s.run_stats()["rounds"]
    assert final == 4
    check_delivery(got, len(ps), tr, infos, final)
    at_end = [k for k, _, i in got if i.rounds == final]
    assert at_end and at_end == sorted(at_end)
    assert [k for k, _, _ in got[-len(at_end):]] == at_end
    s.close()


def test_replanning(batch):
    builders = [obstacle_scenario(k) for k in range(32)]
    ps = [b.build() for b in builders]
    ref = P.Solver()
    ref.upload(ps, gap_tol=GAP, time_limit=60)
    ref.run()
    xs, _ = ref.fetch()
    nxt = [advance_obstacle_scenario(b, p, x).build() for b, p, x in zip(builders, ps, xs)]
    ref.upload_replan(nxt, gap_tol=GAP, time_limit=60)
    ref.run()
    tr0, in0 = ref.fetch_compact()
    s = P.Solver()
    s.upload(ps, gap_tol=GAP, time_limit=60)
    s.run()
    s.upload_replan(nxt, gap_tol=GAP, time_limit=60)
    got = stream(s)
    tr, infos = s.fetch_compact()
    check_delivery(got, len(nxt), tr, infos, s.run_stats()["rounds"])
    for k in range(len(nxt)):
        assert np.array_equal(tr[k], tr0[k])
        assert_info(infos[k], in0[k], skip=("seconds",))
    ref.close(); s.close()


def test_solution_pool(batch):
    ps = batch[:64] + batch[NPLANS:]

    def pools(s):
        return [[(e.search_value, e.uid, e.converged, e.round, e.objective, e.max_violation, e.x.tobytes(), e.traj.tobytes())
                 for e in s.pool(k)] for k in range(len(ps))]

    a = P.Solver(solution_pool=8)
    a.upload(ps, gap_tol=GAP, time_limit=60)
    a.run()
    b = P.Solver(solution_pool=8)
    b.upload(ps, gap_tol=GAP, time_limit=60)
    stream(b)
    assert np.array_equal(a.pool_sizes(), b.pool_sizes())
    assert pools(a) == pools(b)
    a.close(); b.close()


def test_generator_and_callback_exception(batch):
    ps = batch[:32] + batch[NPLANS:]
    s = P.Solver()
    seen = [k for k, t, i in s.solve_batch_streaming(ps, gap_tol=GAP, time_limit=60)]
    assert sorted(seen) == list(range(len(ps)))
    tr, infos = s.fetch_compact()
    calls = []

    def bad(k, t, i):
        calls.append(k)
        if len(calls) == 3:
            raise RuntimeError("controller failed")

    s.upload(ps, gap_tol=GAP, time_limit=60)
    with pytest.raises(RuntimeError, match="controller failed"):
        s.run_streaming(bad)
    assert len(calls) == 3
    tr1, in1 = s.fetch_compact()                  # the run went to its end
    for k in range(len(ps)):
        assert np.array_equal(tr[k], tr1[k])
    s.upload(ps[:8], gap_tol=GAP, time_limit=60)   # and the solver takes the next batch
    s.run()
    _, in2 = s.fetch_compact()
    assert all(i.status == 0 for i in in2)
    # abandoning the generator: the run ends before close() returns
    gen = s.solve_batch_streaming(ps, gap_tol=GAP, time_limit=60)
    next(gen)
    gen.close()
    _, in3 = s.fetch_compact()
    assert len(in3) == len(ps)
    s.close()


def test_pipelined_solver_on_plan(batch):
    batches = [[obstacle_scenario(100 + 40 * j + k).build() for k in range(40)] for j in range(4)]
    ps = P.PipelinedSolver(depth=2)
    want = []
    for b, (tr, infos) in zip(batches, ps.solve_stream_compact([ps.prepare(b, gap_tol=GAP, time_limit=60) for b in batches])):
        want.append(([t.copy() for t in tr], [P.Solver._info(i) for i in infos]))
    got = {}

    def on_plan(bi, k, t, i):
        assert (bi, k) not in got
        got[(bi, k)] = (t, i)

    out = ps.solve_stream_compact([ps.prepare(b, gap_tol=GAP, time_limit=60) for b in batches], on_plan=on_plan)
    assert sorted(got) == [(j, k) for j in range(len(batches)) for k in range(40)]
    for j, (tr, infos) in enumerate(out):
        for k in range(40):
            assert np.array_equal(tr[k], want[j][0][k])
            assert np.array_equal(got[(j, k)][0], tr[k])
            ik = P.Solver._info(infos[k])
            assert_info(got[(j, k)][1], ik)
            assert_info(ik, want[j][1][k], skip=("seconds",))
    ps.close()


def test_errors():
    lib = P.load_library()
    s = P.Solver()
    null_cb = capi.PLAN_DONE()
    ms = C.c_float()
    assert lib.miqp_b200_batch_run_streaming(s._h, capi.PLAN_DONE(lambda *a: None), None, C.byref(ms)) == -2   # no upload
    s.upload([obstacle_scenario(0).build()], gap_tol=GAP, time_limit=60)
    assert lib.miqp_b200_batch_run_streaming(s._h, null_cb, None, C.byref(ms)) == -2
    with pytest.raises(P.MiqpB200Error):
        P.Solver().run_streaming(lambda k, t, i: None)
    got = stream(s)                               # the refused calls left the upload as it was
    assert [k for k, _, _ in got] == [0]
    s.close()
