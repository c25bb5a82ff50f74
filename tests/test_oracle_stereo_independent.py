"""Frame::ComputeStereoMatches: the oracle (orc_stereo_matches) against a second reading written from the reference's
rules (tests/stereo_ref.py), CPU only, so it runs on a clean checkout.  u and z must agree bit for bit on natural
views and on hand-built frames (tests/stereo_cases.py) that put one rule at a time on its edge; the reading's trace
shows that each edge was reached on both sides."""
import functools

import numpy as np
import pytest

from swarmmap_b200 import synth
import oracle_lib
import stereo_cases
import stereo_ref

SF, INV_SF, _, _ = oracle_lib.scale_tables(1.2, 8)


def _planes(ex):
    """mvImagePyramid[l] after operator(): the un-blurred bordered buffer with the level blurred in place."""
    out = []
    for l in range(8):
        buf = ex.level(l, 0).copy()
        buf[19:-19, 19:-19] = ex.level(l, 1)
        out.append(buf)
    return out


def _view(img, nfeat):
    ex = oracle_lib.Extractor(nfeat, 1.2, 8, 20, 7)
    k, d = ex(img)
    return k, d, _planes(ex)


def _both(kl, dl, kr, dr, pl, pr, mbf, mb):
    u0, z0, n0 = oracle_lib.stereo_matches(kl, dl, kr, dr, pl, pr, SF, INV_SF, mbf, mb)
    u1, z1, n1, tr = stereo_ref.stereo_matches(kl, dl, kr, dr, pl, pr, SF, INV_SF, mbf, mb)
    np.testing.assert_array_equal(u1.view(np.uint32), u0.view(np.uint32), err_msg="mvuRight")
    np.testing.assert_array_equal(z1.view(np.uint32), z0.view(np.uint32), err_msg="mvDepth")
    assert n1 == n0
    assert tr["max_abs_delta"] <= 0.5  # the |deltaR| > 1 rule cannot fire (stereo_ref docstring)
    return u1, n1, tr


@pytest.mark.parametrize("w,h,nfeat,seed,kw,mbf,fx", [
    (752, 480, 1000, 1, {}, 47.90639384423901, 458.654),
    (752, 480, 1000, 2, {"d_near": 9.0, "d_far": 0.0}, 47.90639384423901, 458.654),
    (640, 400, 1500, 3, {"right_shift": 6}, 40.0, 400.0),
    (1241, 376, 2000, 4, {"d_near": 70.0, "d_far": 2.0}, 386.1448, 718.856),
    (752, 480, 800, 5, {"d_near": 30.0, "d_far": 25.0}, 47.9, 2000.0),        # maxD > image width
])
def test_natural_views_equal_oracle(w, h, nfeat, seed, kw, mbf, fx):
    left, right = synth.make_stereo_pair(w, h, seed, **kw)
    (kl, dl, pl), (kr, dr, pr) = _view(left, nfeat), _view(right, nfeat)
    u, n, tr = _both(kl, dl, kr, dr, pl, pr, mbf, mbf / fx)
    t = stereo_ref.tally(tr)
    assert n > 200 and t["th_high"] > 0 and t["sad_edge"] > 0 and t["filtered"] > 0, t


def test_identical_views_clear_everything():
    """SAD 0 at every match: the median is 0, and `s < 2.1 * 0` holds for no match."""
    left, _ = synth.make_stereo_pair(752, 480, 6)
    (kl, dl, pl) = _view(left, 1000)
    u, n, tr = _both(kl, dl, kl, dl, pl, pl, 47.9, 47.9 / 458.654)
    t = stereo_ref.tally(tr)
    assert tr["median"] == 0 and n == 0 and (u == -1).all() and t["filtered"] > 400, t


def test_empty_and_flat_right_views():
    left, right = synth.make_stereo_pair(752, 480, 7)
    (kl, dl, pl) = _view(left, 1000)
    kr, dr, pr = _view(right, 1000)
    u, n, tr = _both(kl, dl, kr[:0], dr[:0], pl, pr, 47.9, 47.9 / 458.654)
    assert n == 0 and (tr["outcome"] == stereo_ref.NO_CANDIDATE).all()
    flat = _planes_flat(pr)
    u, n, tr = _both(kl, dl, kr, dr, pl, flat, 47.9, 47.9 / 458.654)
    # a flat right view gives 11 equal SADs: the first minimum is at incR = -5
    reached = tr["bestk"] >= 0
    assert reached.sum() > 100 and (tr["bestk"][reached] == 0).all() and n == 0


def _planes_flat(planes):
    return [np.full_like(p, 128) for p in planes]


@functools.lru_cache(maxsize=None)
def _pair_planes(items):
    left, right = stereo_cases.make_pair(**dict(items))
    return _view(left, 1000)[2], _view(right, 1000)[2]


@functools.lru_cache(maxsize=None)
def _cases():
    out = []
    for c in stereo_cases.build_cases(SF):
        pl, pr = _pair_planes(tuple(sorted(c.pair.items())))
        if c.needs_planes:
            c.needs_planes(c, pl, pr, SF, INV_SF)
        out.append((c, pl, pr))
    return out


def _names():
    return [c.name for c in stereo_cases.build_cases(SF)]


@pytest.mark.parametrize("name", _names())
def test_hand_built_case(name):
    c, pl, pr = next(x for x in _cases() if x[0].name == name)
    kl, dl, kr, dr = c.arrays()
    for call, (mbf, mb) in enumerate(stereo_cases.CALLS):
        u, n, tr = _both(kl, dl, kr, dr, pl, pr, mbf, mb)
        got = {i: stereo_ref.OUTCOMES[tr["outcome"][i]] for i in c.expect[call]}
        assert got == c.expect[call], (call, got)
        if call == 0:
            _check_edges(c, kl, kr, u, tr)


def _check_edges(c, kl, kr, u, tr):
    """The intended edge of each case, read from the trace."""
    if c.name == "tie":
        for i, j in c.tie_cases:
            assert tr["tie"][i] and tr["idx_r"][i] == j
        for i, j in c.no_tie:
            assert not tr["tie"][i] and tr["idx_r"][i] == j
    elif c.name == "th_high":
        assert list(tr["dist"][:2]) == [99, 100]
    elif c.name == "rows":
        r = np.float32(2) * SF[1]
        for i, row, dy in c.row_edges:
            ry = kr["y"][kr["octave"] == 1][i]
            edge = int(np.floor(ry - r)) if dy > 0 else int(np.ceil(ry + r))
            assert edge == (row if abs(dy) < 3 else row + (1 if dy > 0 else -1))
    elif c.name == "u_range":
        assert tr["idx_r"][0] >= 0 and tr["idx_r"][2] >= 0  # uL + 3 and uL - maxD are inside the band
    elif c.name == "window":
        s = tr["scaled_ur0"]
        assert s[0] == -1
        assert sorted(set(s[1:13].astype(int))) == [0, 1, 9, 10]
        assert list(s[13:15].astype(int)) == [stereo_cases.W - 12, stereo_cases.W - 11]
        assert tr["border"][1:10].all() and not tr["border"][10:13].any() and tr["border"][15:19].all()
        assert (tr["outcome"][15:19] == stereo_ref.KEPT).all()  # border rows read inside the chosen SAD windows
    elif c.name == "clamp":
        assert (tr["outcome"][:6] == stereo_ref.CLAMPED).sum() >= 4  # symmetry columns: disparity exactly 0
        assert c.near_zero >= 1, "no left keypoint found whose clamp differs between float and double"
        for i in range(len(kl) - c.near_zero, len(kl)):  # (added last, by clamp_near_zero)
            x = np.float32(kl["x"][i])
            assert u[i] == np.float32(np.float64(x) - 0.01) and u[i] != x - np.float32(0.01)
    elif c.name == "max_disparity":
        assert (tr["disparity"][:3] == 1).all()
    elif c.name == "median_ties":
        s = tr["sad"]
        assert s[0] == s[1] and s[2] == s[3] and s[2] >= 2.1 * s[0] and tr["median"] == s[2]
    elif c.name == "sad_ties":
        assert (tr["n_sad_min"] >= 2).any() and (tr["outcome"] == stereo_ref.KEPT).any()
