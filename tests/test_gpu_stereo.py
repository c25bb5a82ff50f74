"""Frame::ComputeStereoMatches on the GPU (swm_orb_stereo_match, csrc/stereo.cuh) against the oracle
(orc_stereo_matches, itself pinned to the reference's own body in tests/test_ref_stereo.py) and against the second
reading of tests/stereo_ref.py.  The oracle is fed the
GPU extractor's own keypoints, descriptors and pyramid (blurred in place inside its un-blurred border), so the comparison isolates the stereo stage:
mvuRight and mvDepth must be bit-identical floats."""
import numpy as np
import pytest

from swarmmap_b200 import synth
import stereo_ref

pytestmark = pytest.mark.gpu


def _composite(ex, f, l):
    """mvImagePyramid[l] after operator(): the bordered un-blurred buffer with the level blurred in place."""
    buf = ex.debug_plane(f, l, 0).copy()
    buf[19:-19, 19:-19] = ex.debug_plane(f, l, 1)
    return buf


def _pairs(w, h, seeds, **kw):
    lefts, rights = [], []
    for s in seeds:
        l, r = synth.make_stereo_pair(w, h, s, **kw)
        lefts.append(l)
        rights.append(r)
    return np.stack(lefts), np.stack(rights)


@pytest.mark.parametrize("w,h,nfeat,kw,mbf,fx", [
    (752, 480, 1000, {}, 47.90639384423901, 458.654),
    (752, 480, 1000, {"d_near": 9.0, "d_far": 0.0}, 47.90639384423901, 458.654),
    (640, 400, 1500, {"right_shift": 6}, 40.0, 400.0),
    (1241, 376, 2000, {"d_near": 70.0, "d_far": 2.0}, 386.1448, 718.856),
    (752, 480, 800, {"d_near": 30.0, "d_far": 25.0}, 47.9, 2000.0),   # maxD = 2000 > image width: wide search band
])
def test_stereo_matches_equal_oracle(oracle, swm, w, h, nfeat, kw, mbf, fx):
    from swarmmap_b200.orb import ORBextractor
    B = 3
    lefts, rights = _pairs(w, h, (11, 12, 13), **kw)
    exl = ORBextractor(nfeat, 1.2, 8, 20, 7, max_batch=B)
    exr = ORBextractor(nfeat, 1.2, 8, 20, 7, max_batch=B)
    kl, dl, nl = exl.extract_batch(lefts)
    kr, dr, nr = exr.extract_batch(rights)
    mb = mbf / fx
    u, z = exl.stereo_match(exr, mbf, mb, B)
    sf, inv_sf, _, _ = oracle.scale_tables(1.2, 8)
    total = 0
    for f in range(B):
        pl = [_composite(exl, f, l) for l in range(8)]
        pr = [_composite(exr, f, l) for l in range(8)]
        u0, z0, n0 = oracle.stereo_matches(kl[f, :nl[f]], dl[f, :nl[f]], kr[f, :nr[f]], dr[f, :nr[f]], pl, pr, sf, inv_sf, mbf, mb)
        np.testing.assert_array_equal(u[f, :nl[f]].view(np.uint32), u0.view(np.uint32), err_msg=f"mvuRight frame {f}")
        np.testing.assert_array_equal(z[f, :nl[f]].view(np.uint32), z0.view(np.uint32), err_msg=f"mvDepth frame {f}")
        u1, z1, n1, _ = stereo_ref.stereo_matches(kl[f, :nl[f]], dl[f, :nl[f]], kr[f, :nr[f]], dr[f, :nr[f]], pl, pr, sf,
                                                  inv_sf, mbf, mb)
        np.testing.assert_array_equal(u[f, :nl[f]].view(np.uint32), u1.view(np.uint32), err_msg=f"reading frame {f}")
        np.testing.assert_array_equal(z[f, :nl[f]].view(np.uint32), z1.view(np.uint32), err_msg=f"reading frame {f}")
        assert n1 == n0
        total += n0
    assert total > 100 * B


def test_stereo_rejects_mismatched_extractors(swm):
    from swarmmap_b200.orb import ORBextractor
    from swarmmap_b200._lib import SwmError
    a = ORBextractor(500, 1.2, 8, 20, 7, max_batch=1)
    b = ORBextractor(500, 1.2, 8, 20, 7, max_batch=1)
    with pytest.raises(SwmError):
        a.stereo_match(b, 40.0, 0.1, 1)  # nothing extracted yet
    l, r = synth.make_stereo_pair(752, 480, 3)
    a.extract_batch(l[None])
    b.extract_batch(r[None][:, :400, :640].copy())
    with pytest.raises(SwmError):
        a.stereo_match(b, 40.0, 0.1, 1)  # different frame sizes
