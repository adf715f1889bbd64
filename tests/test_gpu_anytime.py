"""Anytime runs (miqp_b200_batch_run_anytime / Solver.run_anytime) and stop requests (miqp_b200_request_stop): every improved
incumbent reaches the caller while the search goes on, the last one of a plan is the result batch_fetch_compact gives for it
after the run, a run without stops computes what batch_run computes, and a stop ends a plan at the select the ABI promises.
The batches mix single-car plans (warp-team node kernel) and multi-car plans (CTA-per-node kernel)."""
import threading
import time

import numpy as np
import pytest

import planner_miqp_b200 as P
from planner_miqp_b200.scenarios import obstacle_scenario, parallel_lanes, two_agent_merge, random_scenario

pytestmark = pytest.mark.gpu

GAP = 1e-4
NPLANS = 256
NMULTI = 48
INFO_FIELDS = ("status", "proven", "objective", "best_bound", "gap", "seconds", "max_violation", "nodes", "qp_iters", "rounds",
               "uncertified", "pool_exhausted")


@pytest.fixture(scope="module")
def batch(testcase_problem):
    return ([obstacle_scenario(k).build() for k in range(NPLANS)] + [testcase_problem]
            + [parallel_lanes(2, nr_steps=5).build(), two_agent_merge(0, nr_steps=8).build(), two_agent_merge(1, nr_steps=8).build()])


@pytest.fixture(scope="module")
def multi():
    """config-4 style: 1-4 cars, time-limited (most multi-car plans run to their limit)"""
    return [random_scenario(k).build() for k in range(NMULTI)]


def same(a, b):
    """bit-identical values (NaN included)"""
    if isinstance(a, float) or isinstance(b, float):
        return np.float64(a).tobytes() == np.float64(b).tobytes()
    return a == b


def assert_info(a, b, skip=("rounds",)):
    for f in INFO_FIELDS:
        if f not in skip:
            assert same(getattr(a, f), getattr(b, f)), (f, getattr(a, f), getattr(b, f))


def anytime(s, stop=lambda k, inc: False, on_done=True):
    """one anytime run: records per plan, and the sequence of callbacks ("inc" / "done", k)"""
    recs, seq, done = {}, [], {}

    def on_inc(k, t, inc):
        recs.setdefault(k, []).append((t, inc))
        seq.append(("inc", k, inc.round))
        return stop(k, inc)

    def on_plan(k, t, info):
        done[k] = (t, info)
        seq.append(("done", k, info.rounds))

    ms = s.run_anytime(on_inc, on_plan if on_done else None)
    assert ms > 0
    return recs, seq, done


def check_records(recs, tr, infos):
    """the last record of every plan with an incumbent is its fetched result; keys fall, rounds rise, all feasible"""
    for k, info in enumerate(infos):
        if info.status != 0:
            assert k not in recs, k
            continue
        assert k in recs, k
        t, inc = recs[k][-1]
        assert np.array_equal(t, tr[k]), k
        assert same(inc.objective, info.objective) and same(inc.max_violation, info.max_violation), (k, inc, info)
        assert inc.search_value >= inc.best_bound
        # the incumbent's key (value, uid) falls strictly: an equal value comes with a smaller uid (the search's tie break)
        keys = [(i.search_value, i.uid) for _, i in recs[k]]
        rounds = [i.round for _, i in recs[k]]
        assert all(a > b for a, b in zip(keys, keys[1:])), (k, keys)
        assert all(a < b for a, b in zip(rounds, rounds[1:])), (k, rounds)
        assert rounds[0] >= 1
        for _, i in recs[k]:
            assert i.max_violation <= 1e-6, (k, i)
            assert i.nodes > 0 and i.seconds > 0


def check_order(seq):
    """within a delivery k ascends (incumbents and plans separately); a plan's incumbents come before its on_done"""
    finished = set()
    for ev, k, _ in seq:
        if ev == "inc":
            assert k not in finished, k
        else:
            finished.add(k)
    for a, b in zip(seq, seq[1:]):
        if a[0] == b[0] == "inc" and a[2] == b[2]:
            assert a[1] < b[1], (a, b)


@pytest.fixture(scope="module")
def plain(batch):
    s = P.Solver(solution_pool=8)
    s.upload(batch, gap_tol=GAP, time_limit=60)
    s.run()
    xs, full = s.fetch()
    tr, infos = s.fetch_compact()
    st = s.run_stats()
    pools = [[(e.search_value, e.uid, e.objective, e.x.tobytes()) for e in s.pool(k)] for k in range(len(batch))]
    s.close()
    return xs, full, tr, infos, st, pools


def test_exact_records_and_unchanged_results(batch, plain):
    xs0, full0, tr0, infos0, st0, pools0 = plain
    s = P.Solver(solution_pool=8)
    s.upload(batch, gap_tol=GAP, time_limit=60)
    recs, seq, done = anytime(s)
    xs, full = s.fetch()
    tr, infos = s.fetch_compact()
    st = s.run_stats()
    check_records(recs, tr, infos)
    check_order(seq)
    assert sorted(done) == list(range(len(batch)))
    for k in range(len(batch)):
        assert np.array_equal(done[k][0], tr[k])
        assert_info(done[k][1], infos[k])
    # the same results as batch_run: vectors, infos, rounds, counters, pool
    assert st["rounds"] == st0["rounds"] and st["nodes"] == st0["nodes"] and st["qp_iters"] == st0["qp_iters"]
    for k in range(len(batch)):
        assert np.array_equal(xs[k], xs0[k]), k
        assert np.array_equal(tr[k], tr0[k]), k
        assert_info(full[k], full0[k], skip=("seconds",))
        assert_info(infos[k], infos0[k], skip=("seconds",))
    assert [[(e.search_value, e.uid, e.objective, e.x.tobytes()) for e in s.pool(k)] for k in range(len(batch))] == pools0
    assert all(v == -1 for v in s.stopped())
    assert sum(len(v) for v in recs.values()) >= len(recs)
    # a plain run after an anytime run is a plain run again
    s.run()
    xs1, _ = s.fetch()
    assert all(np.array_equal(a, b) for a, b in zip(xs1, xs0))
    s.close()


def test_time_limited_multi_car_batch(multi):
    s = P.Solver()
    s.upload(multi, gap_tol=GAP, time_limit=1.0)
    recs, seq, done = anytime(s)
    tr, infos = s.fetch_compact()
    check_records(recs, tr, infos)
    check_order(seq)
    for k in range(len(multi)):
        assert_info(done[k][1], infos[k])
    # without on_done
    s.upload(multi[:8], gap_tol=GAP, time_limit=0.5)
    recs, seq, done = anytime(s, on_done=False)
    assert not done
    tr, infos = s.fetch_compact()
    check_records(recs, tr, infos)
    s.close()


def stop_even(batch):
    s = P.Solver()
    s.upload(batch, gap_tol=GAP, time_limit=60)
    first = {}

    def stop(k, inc):
        first.setdefault(k, inc.round)
        return k % 2 == 0

    recs, seq, done = anytime(s, stop)
    tr, infos = s.fetch_compact()
    xs, _ = s.fetch()
    out = (recs, first, s.stopped(), tr, infos, xs)
    s.close()
    return out


def test_stop_from_the_callback(batch, plain):
    _, _, _, infos0, _, _ = plain
    recs, first, stopped, tr, infos, xs = stop_even(batch)
    check_records(recs, tr, infos)
    n_stopped = 0
    for k in range(len(batch)):
        if k % 2 == 0 and k in first:
            r = first[k]
            assert stopped[k] in (r + 2, -1), (k, r, stopped[k])
            if stopped[k] >= 0:
                n_stopped += 1
                assert all(i.round <= stopped[k] for _, i in recs[k]), k
            assert infos[k].status == 0
            t, inc = recs[k][-1]
            assert np.array_equal(t, tr[k]) and same(inc.objective, infos[k].objective)
        else:
            assert stopped[k] == -1, k
            if infos0[k].proven:
                assert infos[k].proven, k
                assert abs(infos[k].objective - infos0[k].objective) <= 2e-4 * abs(infos0[k].objective), k
    assert n_stopped > 0
    # the same policy again: the same results
    recs2, first2, stopped2, tr2, infos2, xs2 = stop_even(batch)
    assert np.array_equal(stopped, stopped2) and first == first2

    def key(rs):
        return [(t.tobytes(), i.search_value, i.objective, i.round, i.nodes, i.uid) for t, i in rs]

    for k in range(len(batch)):
        assert np.array_equal(xs[k], xs2[k]) and np.array_equal(tr[k], tr2[k])
        assert_info(infos[k], infos2[k], skip=("seconds",))
        assert key(recs.get(k, [])) == key(recs2.get(k, [])), k


def test_stop_before_the_run(batch, multi):
    ps = batch[:16] + batch[NPLANS:] + multi[:8]
    s = P.Solver()
    s.upload(ps, gap_tol=GAP, time_limit=60)
    s.request_stop(3)
    s.request_stop(len(ps) - 1)
    with pytest.raises(P.MiqpB200Error):
        s.request_stop(len(ps))
    recs, _, done = anytime(s)
    _, infos = s.fetch_compact()
    stopped = s.stopped()
    for k in (3, len(ps) - 1):
        assert stopped[k] == 0 and infos[k].nodes == 0 and infos[k].status == 3 and k not in recs, (k, infos[k])
        assert done[k][1].status == 3
    assert all(stopped[k] == -1 for k in range(len(ps)) if k not in (3, len(ps) - 1))
    # requests are cleared when the run ends: the next run searches every plan
    s.run()
    _, infos = s.fetch_compact()
    assert all(i.nodes > 0 for i in infos) and all(v == -1 for v in s.stopped())
    # and at every upload
    s.request_stop(-1)
    s.upload(ps, gap_tol=GAP, time_limit=60)
    s.run()
    assert all(v == -1 for v in s.stopped())
    s.close()


def test_stop_everything_from_the_callback(multi):
    s = P.Solver()
    s.upload(multi, gap_tol=GAP, time_limit=60)
    first = []

    def on_inc(k, t, inc):
        if not first:
            first.append(inc.round)
            s.request_stop(-1)

    s.run_anytime(on_inc)
    r = first[0]
    _, infos = s.fetch_compact()
    stopped = s.stopped()
    assert s.run_stats()["rounds"] == r + 3
    assert all(v in (r + 2, -1) for v in stopped), (r, stopped)
    assert (stopped == r + 2).sum() > 0
    assert all(i.status in (0, 3) for i in infos)
    s.close()


def test_stop_from_another_thread(multi):
    s = P.Solver()
    s.upload(multi, gap_tol=GAP, time_limit=60)
    woken = threading.Event()
    first = []

    def stopper():
        woken.wait(120)
        s.request_stop(-1)

    th = threading.Thread(target=stopper)
    th.start()

    def on_inc(k, t, inc):
        if not first:
            first.append(inc.round)
            woken.set()

    t0 = time.perf_counter()
    s.run_anytime(on_inc)
    wall = time.perf_counter() - t0
    th.join()
    r = first[0]
    _, infos = s.fetch_compact()
    stopped = s.stopped()
    assert wall < 20.0, wall
    hit = stopped[stopped >= 0]
    assert len(hit) > 0 and (hit >= r + 2).all() and len(set(hit.tolist())) == 1, (r, stopped)
    assert all(i.status in (0, 3) for i in infos)
    s.close()


def test_errors(batch):
    import ctypes as C
    from planner_miqp_b200 import capi
    lib = P.load_library()
    s = P.Solver()
    ms = C.c_float()
    noop = capi.INCUMBENT_FOUND(lambda *a: 0)
    assert lib.miqp_b200_batch_run_anytime(s._h, noop, capi.PLAN_DONE(), None, C.byref(ms)) == -2   # no upload
    assert lib.miqp_b200_request_stop(s._h, 0) == -2
    s.upload(batch[:4], gap_tol=GAP, time_limit=60)
    assert lib.miqp_b200_stopped(s._h, (C.c_int * 4)()) == -2                                         # before a run
    assert lib.miqp_b200_batch_run_anytime(s._h, capi.INCUMBENT_FOUND(), capi.PLAN_DONE(), None, C.byref(ms)) == -2
    assert lib.miqp_b200_request_stop(s._h, 4) == -2 and lib.miqp_b200_request_stop(s._h, -2) == -2
    recs, _, _ = anytime(s, on_done=False)          # the refused calls left the upload as it was
    assert sorted(recs) == [0, 1, 2, 3]
    s.close()
