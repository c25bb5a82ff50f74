"""Pins the isInFrustum / PredictScale oracle (oracle/orb_oracle_frustum.cpp) to the REFERENCE'S OWN bodies of
Frame::isInFrustum (Frame.cc:316-375) and MapPoint::PredictScale (MapPoint.cc:476-485), compiled by `make -C oracle ref`
on the test doubles of tests/ref_matcher_lib.py.  Skips where the reference sources are absent; on a clean checkout
tests/test_oracle_frustum_independent.py pins the oracle to the independent reading instead."""
import numpy as np
import pytest

import frustum_cases as FC
import oracle_frustum_lib as O
import ref_matcher_lib as R
from swarmmap_b200.matcher import Frame

pytestmark = pytest.mark.skipif(not R.available(), reason="needs oracle/_ref/liborbmatcher_ref.so, compiled by `make -C oracle ref` "
                                                          "from the reference project's sources, which the repository does not contain")


def _ref(sc):
    scales = R.Scales(1.2, 8)
    scales.log_sf = float(FC.LOG_SF)
    b = sc["bounds4"]
    f = Frame([float(b[0])], [float(b[2])], [0], [0.0], np.zeros((1, 32), np.uint8), (b[0], b[2], b[1], b[3]), FC.SF)
    T = np.eye(4, dtype=np.float32)
    T[:3, :4] = sc["T"]
    rf, kf = R.frame(f, scales, K=sc["K"], Tcw=T)
    rp, kp = R.points(sc["pos"], np.zeros((len(sc["pos"]), 32), np.uint8), normal=sc["normal"], min_dist=sc["min_d"],
                      max_dist=sc["max_d"])
    return R.is_in_frustum(rf, rp, 0.5)


@pytest.mark.parametrize("which", ["random", "kitti", "edges"])
def test_is_in_frustum_equals_reference(which):
    rng = np.random.default_rng(3)
    if which == "random":
        sc = FC.random_scene(rng, 3000)
    elif which == "kitti":
        sc = FC.random_scene(rng, 3000, K=(718.856, 718.856, 607.1928, 185.2157), bounds4=(-31.4, 1272.6, -17.9, 393.3))
    else:
        thr = FC.thresholds_by_bisection(lambda a, b: O.predict_scale(a, b, FC.LOG_SF, 8))
        sc, _ = FC.edge_scene(thr)
    got = _ref(sc)
    o = O.is_in_frustum(sc["T"], sc["K"], sc["bounds4"], sc["pos"], sc["normal"], sc["min_d"], sc["max_d"], FC.LOG_SF, 8)
    assert np.array_equal(got["in_view"], o["in_view"])
    iv = o["in_view"] == 1
    for a, b in (("proj_x", "u"), ("proj_y", "v"), ("view_cos", "view_cos"), ("level", "level")):
        assert FC.same_bits(got[a][iv], o[b][iv]).all(), a


def test_predict_scale_equals_reference_at_every_threshold():
    thr = FC.thresholds_by_bisection(lambda a, b: O.predict_scale(a, b, FC.LOG_SF, 8))
    r = np.concatenate([[FC.down(t), t, FC.up(t)] for t in thr] + [[0.5, 1.0, 1e30]]).astype(np.float32)
    one = np.ones_like(r)
    assert np.array_equal(R.predict_scale(r, one, float(FC.LOG_SF), 8), O.predict_scale(r, one, FC.LOG_SF, 8))
