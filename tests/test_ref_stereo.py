"""Frame::ComputeStereoMatches: the oracle's restatement (oracle/orb_oracle_match.cpp: orc_stereo_matches) against the
REFERENCE'S OWN body (code/src/Frame.cc:516-690, cut at build time and compiled unmodified against the stand-in
cv::Mat / cv::cuda::GpuMat of oracle/ref_shim_matcher, see oracle/ref_orbmatcher_wrap.cpp: refm_stereo_matches).
CPU only: the keypoints, descriptors and pyramids of both views come from the oracle's extractor."""
import numpy as np
import pytest

from swarmmap_b200 import synth
import oracle_lib
import ref_matcher_lib

pytestmark = pytest.mark.skipif(not ref_matcher_lib.available(), reason="needs oracle/_ref/liborbmatcher_ref.so, compiled by `make -C oracle ref` "
                                                                        "from the reference project's sources, which the repository does not contain")


def _views(w, h, nfeat, seed, **kw):
    left, right = synth.make_stereo_pair(w, h, seed, **kw)
    out = []
    for img in (left, right):
        ex = oracle_lib.Extractor(nfeat, 1.2, 8, 20, 7)
        k, d = ex(img)
        planes = []
        for l in range(8):  # mvImagePyramid[l] after operator(): blurred in place inside the un-blurred bordered buffer
            buf = ex.level(l, 0).copy()
            buf[19:-19, 19:-19] = ex.level(l, 1)
            planes.append(buf)
        out.append((k, d, planes))
    return out


@pytest.mark.parametrize("w,h,nfeat,seed,kw,mbf,fx", [
    (752, 480, 1000, 1, {}, 47.90639384423901, 458.654),                       # EuRoC-shaped, ground-plane disparities 4..40 px
    (752, 480, 1000, 2, {"d_near": 9.0, "d_far": 0.0}, 47.90639384423901, 458.654),   # disparities down to 0: the <= 0 clamp
    (640, 400, 1500, 3, {"right_shift": 6}, 40.0, 400.0),                      # partly negative disparities: rejected
    (1241, 376, 2000, 4, {"d_near": 70.0, "d_far": 2.0}, 386.1448, 718.856),   # KITTI-shaped
    (752, 480, 800, 5, {"d_near": 30.0, "d_far": 25.0}, 47.9, 2000.0),          # maxD = 2000 > image width: wide search band
])
def test_oracle_stereo_equals_reference(w, h, nfeat, seed, kw, mbf, fx):
    (kl, dl, pl), (kr, dr, pr) = _views(w, h, nfeat, seed, **kw)
    sf, inv_sf, _, _ = oracle_lib.scale_tables(1.2, 8)
    mb = mbf / fx
    u0, z0, n0 = oracle_lib.stereo_matches(kl, dl, kr, dr, pl, pr, sf, inv_sf, mbf, mb)
    u1, z1, n1 = ref_matcher_lib.stereo_matches(kl, dl, kr, dr, pl, pr, sf, inv_sf, mbf, mb)
    assert n1 > 50, "the case must produce stereo matches"
    assert n0 == n1
    np.testing.assert_array_equal(u0.view(np.uint32), u1.view(np.uint32))  # bit-exact floats, -1 where unmatched
    np.testing.assert_array_equal(z0.view(np.uint32), z1.view(np.uint32))
    ok = u0 >= 0
    # the recovered disparity is the planted one (sanity of the test data, not of the port)
    if not kw.get("right_shift"):
        d_far, d_near = kw.get("d_far", 4.0), kw.get("d_near", 40.0)
        planted = d_far + (d_near - d_far) * kl["y"][ok] / (h - 1)
        assert np.median(np.abs((kl["x"][ok] - u0[ok]) - planted)) < 1.0


def test_oracle_stereo_no_right_keypoints():
    (kl, dl, pl), (kr, dr, pr) = _views(752, 480, 500, 7)
    sf, inv_sf, _, _ = oracle_lib.scale_tables(1.2, 8)
    u0, z0, n0 = oracle_lib.stereo_matches(kl, dl, kr[:0], dr[:0], pl, pr, sf, inv_sf, 47.9, 47.9 / 458.0)
    assert n0 == 0 and (u0 == -1).all() and (z0 == -1).all()
