"""The resident MapPoint table and the two tracking projections run from it (swm_match_local_map*, swm_match_last_frame)
on the device, against the oracle fed by the independent reading (tests/frustum_ref.py) and against the host path the
wrapper used before (the reading's window query passed to swm_match_window_resident on the same frame).

Compared bit for bit: in_view, u, v, view_cos and level of every list entry, the assignment, nmatches and n_to_match."""
import threading

import numpy as np
import pytest

import frustum_cases as FC
import frustum_ref
import oracle_frustum_lib as O
import oracle_lib
from swarmmap_b200 import _lib
from localmap_scenes import _b4_to_frame, make_world, points_kw, resident, upload_table
from swarmmap_b200.matcher import Frame, MapPointTable, ORBmatcher

pytestmark = pytest.mark.gpu

F32 = np.float32
NNRATIO = 0.8


def expect_points(w, m, rf, th, rows=None, frame_rows=None, tab=None):
    """The reading's query -> (oracle match, resident host-path match, track, n_to_match)."""
    tab = tab if tab is not None else w["tab"]
    rows = w["rows"] if rows is None else rows
    fr = w["frame_rows"] if frame_rows is None else frame_rows
    tr, q, blocked, ntm = frustum_ref.local_map_query(tab, rows, fr, w["T"], w["K"], w["b4"], FC.SF, FC.LOG_SF, 8, th)
    # the oracle's isInFrustum on the same list, masked the same way, equals the reading
    o = O.is_in_frustum(w["T"], w["K"], w["b4"], tab["pos"][rows], tab["normal"][rows], tab["min_d"][rows],
                        tab["max_d"][rows], FC.LOG_SF, 8)
    for k in ("in_view", "u", "v", "view_cos", "level"):
        assert FC.same_bits(np.where(tr["in_view"] == 1, o[k], 0).astype(o[k].dtype), tr[k]).all(), k
    args = (q["desc"], q["u"], q["v"], q["radius"], q["min_level"], q["max_level"], q["valid"], q["blocks"], 100, 1)
    n_o, a_o = oracle_lib.match_window(w["F"], *args, NNRATIO, False, tgt_blocked=blocked)
    n_r, a_r = m.match_window(rf, *args, tgt_blocked=blocked, check_ori=False)
    assert n_o == n_r and np.array_equal(a_o, a_r)
    return n_o, a_o, tr, ntm


def check_points(res, exp):
    n, asg, ntm, track = res
    n_o, a_o, tr, ntm_o = exp
    assert n == n_o and ntm == ntm_o
    assert np.array_equal(asg, a_o)
    for k in ("in_view", "u", "v", "view_cos", "level"):
        assert FC.same_bits(track[k], tr[k]).all(), (k, np.nonzero(~FC.same_bits(track[k], tr[k]))[0][:8])


@pytest.fixture(scope="module")
def matcher():
    return ORBmatcher(NNRATIO, True)


@pytest.mark.parametrize("th", [1.0, 3.0, 5.0])
def test_local_map_single_equals_oracle_and_host_path(matcher, th):
    rng = np.random.default_rng(10 + int(th))
    w = make_world(rng, 2000)
    rf, table = resident(w["F"]), upload_table(w["tab"])
    res = matcher.search_local_map(**points_kw(w, rf, table, th))
    exp = expect_points(w, matcher, rf, th)
    check_points(res, exp)
    assert res[0] > 200 and 0 < res[2] < len(w["rows"])


def test_kitti_size(matcher):
    rng = np.random.default_rng(3)
    w = make_world(rng, 3000, K=(718.856, 718.856, 607.1928, 185.2157), b4=(0.0, 1241.0, 0.0, 376.0), extra=1000)
    rf, table = resident(w["F"]), upload_table(w["tab"])
    check_points(matcher.search_local_map(**points_kw(w, rf, table, 1.0)), expect_points(w, matcher, rf, 1.0))


def test_edge_points_through_upsert(matcher):
    """The hand-built edge points of tests/frustum_cases.py, written into a table and projected on the device."""
    thr = np.zeros(7, F32)
    assert _lib.load().swm_predict_scale_thresholds(float(FC.LOG_SF), 8, _lib.ptr(thr)) == 0
    sc, names = FC.edge_scene(thr)
    n = len(names)
    rng = np.random.default_rng(5)
    tab = dict(pos=sc["pos"], normal=sc["normal"], min_d=sc["min_d"], max_d=sc["max_d"],
               desc=rng.integers(0, 256, (n, 32), dtype=np.uint8), has_obs=np.ones(n, np.uint8),
               bad=np.zeros(n, np.uint8))
    b4 = sc["bounds4"]
    kx = rng.uniform(b4[0], b4[1] - 1e-3, 40).astype(F32)
    ky = rng.uniform(b4[2], b4[3] - 1e-3, 40).astype(F32)
    F = Frame(kx, ky, rng.integers(0, 8, 40), rng.uniform(0, 360, 40), rng.integers(0, 256, (40, 32), dtype=np.uint8),
              _b4_to_frame(b4), FC.SF)
    w = dict(T=sc["T"], K=sc["K"], b4=b4, tab=tab, F=F, frame_rows=np.full(40, -1, np.int32),
             rows=np.arange(n, dtype=np.int32))
    rf, table = resident(F), upload_table(tab)
    res = matcher.search_local_map(**points_kw(w, rf, table, 1.0))
    check_points(res, expect_points(w, matcher, rf, 1.0))
    tr = frustum_ref.is_in_frustum(sc["T"], sc["K"], b4, sc["pos"], sc["normal"], sc["min_d"], sc["max_d"], FC.LOG_SF, 8)
    assert set(tr["rule"]) == set(range(len(frustum_ref.RULES)))
    lvl = dict(zip(names, res[3]["level"]))
    for k in range(1, 8):
        assert lvl[f"ratio=thr{k}"] == k - 1 and lvl[f"ratio=thr{k}+1ulp"] == k


def test_batch_128_jobs_equals_singles_shared_and_own_tables(matcher):
    """128 agents at the benchmark's 752x480 geometry, local maps of 2000 points; half the jobs share one table (their
    rows offset into it), the others have a table each; duplicate rows in some lists; batch == singles == oracle."""
    rng = np.random.default_rng(21)
    P = 128
    worlds = [make_world(rng, 2000) for _ in range(P)]
    shared_tab = {k: np.concatenate([w["tab"][k] for w in worlds[:P // 2]]) for k in worlds[0]["tab"]}
    shared = upload_table(shared_tab)
    jobs, exps, rfs, tabs = [], [], [], []
    for a, w in enumerate(worlds):
        rf = resident(w["F"])
        rfs.append(rf)
        if a < P // 2:
            off = 2000 * a
            rows = (w["rows"] + off).astype(np.int32)
            if a % 4 == 1:
                rows = np.concatenate([rows, rows[:50]]).astype(np.int32)  # duplicates keep list order
            fr = np.where(w["frame_rows"] >= 0, w["frame_rows"] + off, -1).astype(np.int32)
            ww = dict(w, rows=rows, frame_rows=fr)
            jobs.append(points_kw(ww, rf, shared, 1.0))
            exps.append(expect_points(ww, matcher, rf, 1.0, tab=shared_tab))
        else:
            t = upload_table(w["tab"])
            tabs.append(t)
            jobs.append(points_kw(w, rf, t, 1.0))
            exps.append(expect_points(w, matcher, rf, 1.0))
    got = matcher.search_local_map_batch(jobs)
    for r, e in zip(got, exps):
        check_points(r, e)
    for a in (0, 1, 5, 64, 127):
        single = matcher.search_local_map(**jobs[a])
        check_points(single, exps[a])
        assert np.array_equal(single[1], got[a][1])
    assert _lib.load().swm_matcher_last_device_ms(matcher._h) > 0


def test_empty_lists_and_frames_bad_and_erased_rows(matcher):
    rng = np.random.default_rng(8)
    w = make_world(rng, 1500)
    rf, table = resident(w["F"]), upload_table(w["tab"])
    # empty list
    n, asg, ntm, track = matcher.search_local_map(**points_kw(w, rf, table, 1.0, rows=np.zeros(0, np.int32)))
    assert n == 0 and ntm == 0 and (asg == -1).all() and len(track["u"]) == 0
    # empty frame: the frustum test still runs, nothing can match
    E = Frame(np.zeros(0), np.zeros(0), np.zeros(0), np.zeros(0), np.zeros((0, 32), np.uint8), w["F"].bounds, FC.SF)
    re = resident(E)
    ww = dict(w, F=E, frame_rows=np.zeros(0, np.int32))
    res = matcher.search_local_map(**points_kw(ww, re, table, 1.0))
    exp = expect_points(ww, matcher, re, 1.0)
    check_points(res, exp)
    assert res[0] == 0 and res[2] > 0
    # erase a third of the points (upsert with bad = 1) and mark them bad in the reading's table as well
    er = rng.choice(1500, 500, replace=False).astype(np.int32)
    tab2 = {k: v.copy() for k, v in w["tab"].items()}
    tab2["bad"][er] = 1
    table.upsert(er, tab2["pos"][er], tab2["normal"][er], tab2["min_d"][er], tab2["max_d"][er], tab2["desc"][er],
                 tab2["has_obs"][er], tab2["bad"][er])
    ww = dict(w, tab=tab2)
    check_points(matcher.search_local_map(**points_kw(ww, rf, table, 1.0)), expect_points(ww, matcher, rf, 1.0))


def test_table_growth_between_calls(matcher):
    """Capacity grows from 16 rows while keeping the contents; a query after an upsert sees it."""
    rng = np.random.default_rng(31)
    w = make_world(rng, 2000)
    rf = resident(w["F"])
    table = MapPointTable(0, 16)
    half = 1000
    t = w["tab"]
    table.upsert(np.arange(half, dtype=np.int32), t["pos"][:half], t["normal"][:half], t["min_d"][:half], t["max_d"][:half],
                 t["desc"][:half], t["has_obs"][:half], t["bad"][:half])
    rows_half = w["rows"][w["rows"] < half]
    fr_half = np.where(w["frame_rows"] < half, w["frame_rows"], -1).astype(np.int32)
    first = matcher.search_local_map(**points_kw(w, rf, table, 1.0, rows=rows_half, frame_rows=fr_half))
    check_points(first, expect_points(w, matcher, rf, 1.0, rows=rows_half, frame_rows=fr_half))
    rest = np.arange(half, 2000, dtype=np.int32)
    table.upsert(rest, t["pos"][rest], t["normal"][rest], t["min_d"][rest], t["max_d"][rest], t["desc"][rest],
                 t["has_obs"][rest], t["bad"][rest])
    assert table.size == 2000
    full = matcher.search_local_map(**points_kw(w, rf, table, 1.0))
    check_points(full, expect_points(w, matcher, rf, 1.0))
    table.upsert(np.arange(2000, dtype=np.int32), -t["pos"], t["normal"], t["min_d"], t["max_d"], t["desc"],
                 t["has_obs"], t["bad"])
    after = matcher.search_local_map(**points_kw(w, rf, table, 1.0))
    assert after[2] < full[2] // 4  # most points are behind the camera now


def _same(res, exp):
    n, asg, ntm, track = res
    n_o, a_o, tr, ntm_o = exp
    return n == n_o and ntm == ntm_o and np.array_equal(asg, a_o) and all(
        FC.same_bits(track[k], tr[k]).all() for k in ("in_view", "u", "v", "view_cos", "level"))


def test_upserts_from_another_thread_while_queries_run(matcher):
    """A second thread keeps upserting while batch queries run: rows past the end, so that the table grows (and its
    block is reallocated) many times, and the queried rows, alternately moved behind the camera and put back.  Every
    query must return exactly the result of one table state -- the one before or the one after a rewrite -- and all
    jobs of one batch the same state: never a mix, never a read of a block that growth has freed."""
    rng = np.random.default_rng(77)
    w = make_world(rng, 2000)
    rf = resident(w["F"])
    t = w["tab"]
    table = upload_table(t, MapPointTable(0, 2048))
    moved = dict(t, pos=(-t["pos"]).astype(F32))
    exp = [expect_points(w, matcher, rf, 1.0), expect_points(dict(w, tab=moved), matcher, rf, 1.0)]
    assert exp[0][3] != exp[1][3]  # the two table states give different n_to_match
    stop, errors, writes = threading.Event(), [], [0]
    filler = dict(pos=np.ones((4096, 3), F32), normal=np.ones((4096, 3), F32), min_d=np.zeros(4096, F32),
                  max_d=np.ones(4096, F32), desc=np.zeros((4096, 32), np.uint8), has_obs=np.ones(4096, np.uint8),
                  bad=np.zeros(4096, np.uint8))
    rows_all = np.arange(2000, dtype=np.int32)

    def writer():
        try:
            end = 2000
            while not stop.is_set():
                if end < 600000:  # grow: each doubling of the capacity reallocates the table's block
                    table.upsert(np.arange(end, end + 4096, dtype=np.int32), filler["pos"], filler["normal"],
                                 filler["min_d"], filler["max_d"], filler["desc"], filler["has_obs"], filler["bad"])
                    end += 4096
                src = moved if writes[0] % 2 == 0 else t
                table.upsert(rows_all, src["pos"], src["normal"], src["min_d"], src["max_d"], src["desc"],
                             src["has_obs"], src["bad"])
                writes[0] += 1
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    th = threading.Thread(target=writer)
    th.start()
    states = []
    try:
        for _ in range(40):
            got = matcher.search_local_map_batch([points_kw(w, rf, table, 1.0)] * 4)
            which = [0 if _same(r, exp[0]) else 1 if _same(r, exp[1]) else -1 for r in got]
            assert -1 not in which and len(set(which)) == 1, which
            states.append(which[0])
    finally:
        stop.set()
        th.join()
    assert not errors, errors
    assert writes[0] > 10 and table.size > 2000 + 4096 * 10
    print(f"{writes[0]} rewrites, table of {table.size} rows, query states {states}")


def test_upsert_and_query_refusals(matcher):
    rng = np.random.default_rng(2)
    w = make_world(rng, 300)
    rf, table = resident(w["F"]), upload_table(w["tab"])
    with pytest.raises(_lib.SwmError):
        table.upsert(np.array([3, -1], np.int32), np.zeros((2, 3)), np.zeros((2, 3)), np.ones(2), np.ones(2),
                     np.zeros((2, 32), np.uint8), np.ones(2))
    assert table.size == 300
    with pytest.raises(_lib.SwmError):  # row past the table
        matcher.search_local_map(**points_kw(w, rf, table, 1.0, rows=np.array([0, 300], np.int32)))
    with pytest.raises(_lib.SwmError):  # frame row past the table
        matcher.search_local_map(**points_kw(w, rf, table, 1.0, frame_rows=np.full(w["F"].N, 300, np.int32)))
    # a row given twice in one upsert takes its last entry
    t2 = MapPointTable()
    t2.upsert(np.array([0, 0], np.int32), np.array([[0, 0, -5], [0, 0, 5]], F32), np.array([[0, 0, 1]] * 2, F32),
              np.zeros(2), np.full(2, 100.0), np.zeros((2, 32), np.uint8), np.ones(2))
    E = Frame([10.0], [10.0], [0], [0.0], np.zeros((1, 32), np.uint8), (0.0, 0.0, 752.0, 480.0), FC.SF)
    T = np.hstack([np.eye(3), np.zeros((3, 1))]).astype(F32)
    r = matcher.search_local_map(F=resident(E), table=t2, Tcw=T, K=FC.K_EUROC, log_scale_factor=FC.LOG_SF,
                                 rows=np.array([0], np.int32), th=1.0, scale_factors=FC.SF)
    assert r[2] == 1


def test_last_frame_equals_oracle_and_host_path(matcher):
    rng = np.random.default_rng(44)
    w = make_world(rng, 2000)
    cur = resident(w["F"])
    # the last frame: the current frame's keypoints moved a little, holding the rows of their points (some outliers)
    F = w["F"]
    L = Frame(F.x + F32(1.5), F.y - F32(0.5), F.octave, F.angle, F.desc, F.bounds, FC.SF)
    last = resident(L)
    last_rows = np.where(rng.random(F.N) < 0.9, w["owner"], -1).astype(np.int32)
    table = upload_table(w["tab"])
    cur_rows = np.full(F.N, -1, np.int32)
    cur_rows[rng.choice(F.N, 30, replace=False)] = rng.integers(0, 2000, 30)
    for th, cr in ((15.0, None), (7.0, cur_rows)):
        n, asg = matcher.search_last_frame(cur, last, table, w["T"], w["K"], FC.LOG_SF, last_rows, cr, th, FC.SF)
        q, blocked = frustum_ref.last_frame_query(w["tab"], last_rows, L.octave, L.angle, cr, w["T"], w["K"], w["b4"],
                                                  FC.SF, th)
        # the oracle's projection equals the reading's
        ok, u, v = O.project_last(w["T"], w["K"], w["b4"], w["tab"]["pos"][np.maximum(last_rows, 0)])
        assert np.array_equal(ok & (last_rows >= 0), q["valid"]) and FC.same_bits(np.where(q["valid"] == 1, u, 0), q["u"]).all()
        args = (q["desc"], q["u"], q["v"], q["radius"], q["min_level"], q["max_level"], q["valid"], q["blocks"], 100, 0)
        n_o, a_o = oracle_lib.match_window(F, *args, NNRATIO, True, angle=q["angle"], tgt_blocked=blocked,
                                           assignment=np.full(F.N, -3, np.int32))
        n_r, a_r = matcher.match_window(cur, *args, angle=q["angle"], tgt_blocked=blocked,
                                        assignment=np.full(F.N, -3, np.int32), check_ori=True)
        assert n == n_o == n_r and n > 100
        assert np.array_equal(asg, a_o) and np.array_equal(asg, a_r)
    # last-frame jobs in a batch with local-map jobs
    got = matcher.search_local_map_batch([
        dict(mode=_lib.LOCALMAP_LAST, F=cur, last=last, table=table, Tcw=w["T"], K=w["K"], log_scale_factor=FC.LOG_SF,
             rows=last_rows, th=15.0, scale_factors=FC.SF),
        points_kw(w, cur, table, 1.0)])
    n1, a1 = matcher.search_last_frame(cur, last, table, w["T"], w["K"], FC.LOG_SF, last_rows, None, 15.0, FC.SF)
    assert got[0][0] == n1 and np.array_equal(got[0][1], a1)
    check_points(got[1], expect_points(w, matcher, cur, 1.0))
