"""Frame::isInFrustum and MapPoint::PredictScale: the oracle (oracle/orb_oracle_frustum.cpp) against a second reading
written from the reference's rules (tests/frustum_ref.py), bit for bit, CPU only.  Random views at the benchmark's
camera and hand-built points that put each rule on its edge (tests/frustum_cases.py); the reading's trace shows that
every outcome occurred.  Also: the level thresholds the device counts instead of calling log (swm_predict_scale_
thresholds) against the oracle, with the monotonicity they rely on checked over 10^6 ulps either side."""
import numpy as np
import pytest

import frustum_cases as FC
import frustum_ref
import oracle_frustum_lib as O

FIELDS = ("in_view", "u", "v", "view_cos", "level")


def _both(sc):
    args = (sc["T"], sc["K"], sc["bounds4"], sc["pos"], sc["normal"], sc["min_d"], sc["max_d"], sc["log_sf"],
            sc["nlevels"])
    o = O.is_in_frustum(*args)
    r = frustum_ref.is_in_frustum(*args)
    for f in FIELDS:
        ok = FC.same_bits(o[f], r[f])
        assert ok.all(), (f, np.nonzero(~ok)[0][:10])
    return r


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5])
def test_random_views_equal_oracle(seed):
    rng = np.random.default_rng(seed)
    r = _both(FC.random_scene(rng, 4000))
    counts = np.bincount(r["rule"], minlength=len(frustum_ref.RULES))
    assert (counts > 0).all(), dict(zip(frustum_ref.RULES, counts))
    assert len(np.unique(r["level"][r["in_view"] == 1])) == FC.NLEVELS


def test_kitti_camera_and_shifted_bounds():
    rng = np.random.default_rng(9)
    sc = FC.random_scene(rng, 3000, K=(718.856, 718.856, 607.1928, 185.2157), bounds4=(-31.4, 1272.6, -17.9, 393.3))
    _both(sc)


def _edge():
    thr = FC.thresholds_by_bisection(lambda a, b: O.predict_scale(a, b, FC.LOG_SF, FC.NLEVELS))
    return FC.edge_scene(thr), thr


def test_edges_equal_oracle_and_every_outcome_occurs():
    (sc, names), thr = _edge()
    r = _both(sc)
    rule = {n: frustum_ref.RULES[k] for n, k in zip(names, r["rule"])}
    lvl = dict(zip(names, r["level"]))
    expect = {"z=+0": "in_view", "z=-0": "u_out", "z=-1ulp": "behind",
              "u=min": "in_view", "u=min-1ulp": "u_out", "u=max": "in_view", "u=max+1ulp": "u_out",
              "v=min": "in_view", "v=min-1ulp": "v_out", "v=max": "in_view", "v=max+1ulp": "v_out",
              "dist=min": "in_view", "dist=min-1ulp": "dist_small", "dist=min+1ulp": "in_view",
              "dist=max": "in_view", "dist=max+1ulp": "dist_large", "dist=max-1ulp": "in_view",
              "cos=0.5": "in_view", "cos=0.5-1ulp": "angle", "cos=0.998f": "in_view", "cos=0.998f-1ulp": "in_view"}
    for n, e in expect.items():
        assert rule[n] == e, (n, rule[n], e)
    assert set(rule.values()) == set(frustum_ref.RULES)
    # z = +0: u is NaN and passes (as in the reference); the ratio is inf -> the top level
    i = names.index("z=+0")
    assert np.isnan(r["u"][i]) and lvl["z=+0"] == FC.NLEVELS - 1
    for k in range(1, FC.NLEVELS):
        assert lvl[f"ratio=thr{k}"] == k - 1 and lvl[f"ratio=thr{k}-1ulp"] == k - 1 and lvl[f"ratio=thr{k}+1ulp"] == k
    assert lvl["ratio=0.9"] == 0 and lvl["ratio=1"] == 0 and lvl["ratio=1e30"] == FC.NLEVELS - 1
    # RadiusByViewingCos compares with the double 0.998: 0.998f is above it, the float below it is not
    vc = dict(zip(names, r["view_cos"]))
    for th in (1.0, 3.0, 5.0):
        rad = frustum_ref.radius_by_viewing_cos([vc["cos=0.998f"], vc["cos=0.998f-1ulp"], vc["cos=0.5"]], th)
        base = np.array([2.5, 4.0, 4.0], np.float32)
        assert np.array_equal(rad, base if th == 1.0 else base * np.float32(th))


def test_last_frame_projection_equals_oracle():
    rng = np.random.default_rng(4)
    sc = FC.random_scene(rng, 4000)
    (es, _), _ = _edge()
    for s in (sc, es):
        o = O.project_last(s["T"], s["K"], s["bounds4"], s["pos"])
        r = frustum_ref.project_last(s["T"], s["K"], s["bounds4"], s["pos"])
        for a, b in zip(o, r):
            assert FC.same_bits(a, b).all()
    assert 0 < o[0].sum() < len(o[0])


def test_predict_scale_thresholds_are_exact(swm):
    """The device counts the thresholds a ratio exceeds.  The library's thresholds equal the oracle's boundaries, and
    the oracle's level is monotone over 10^6 ulps on both sides of each, so the count equals PredictScale."""
    lib = swm.load()
    for scale_factor, nlevels in ((1.2, 8), (1.2, 12), (1.5, 4), (2.0, 2)):
        _, log_sf = FC.scale_tables(scale_factor, nlevels)
        thr = np.zeros(nlevels - 1, np.float32)
        assert lib.swm_predict_scale_thresholds(float(log_sf), nlevels, swm.ptr(thr)) == 0
        ref = FC.thresholds_by_bisection(lambda a, b: O.predict_scale(a, b, log_sf, nlevels), log_sf, nlevels)
        assert np.array_equal(thr.view(np.uint32), ref.view(np.uint32)), (thr, ref)
        for k, t in enumerate(thr, 1):
            bits = np.int64(np.array([t], np.float32).view(np.uint32)[0]) + np.arange(-10 ** 6, 10 ** 6 + 1)
            r = bits.astype(np.uint32).view(np.float32)
            lv = O.predict_scale(r, np.ones_like(r), log_sf, nlevels)
            assert (np.diff(lv) >= 0).all()
            count = (r[:, None] > thr[None, :]).sum(1)
            assert np.array_equal(lv, count), k
            assert lv[10 ** 6] == k - 1 and lv[10 ** 6 + 1] == k
    assert lib.swm_predict_scale_thresholds(float(FC.LOG_SF), 0, swm.ptr(thr)) == -1
    assert lib.swm_predict_scale_thresholds(float(FC.LOG_SF), 17, swm.ptr(thr)) == -1
    assert lib.swm_predict_scale_thresholds(0.0, 8, swm.ptr(thr)) == -1
    assert lib.swm_predict_scale_thresholds(float(FC.LOG_SF), 8, None) == -1
