"""Pins the oracle's matchers (oracle/orb_oracle_match.cpp) to the REFERENCE'S OWN code: code/src/ORBmatcher.cc compiled
UNMODIFIED (oracle/_ref/liborbmatcher_ref.so, `make -C oracle ref`) together with the reference's own bodies of
Frame::AssignFeaturesToGrid / GetFeaturesInArea / PosInGrid / isInFrustum, KeyFrame::GetFeaturesInArea / IsInImage and
MapPoint::PredictScale, on test doubles of Frame / KeyFrame / MapPoint.

Every test builds one scene, runs the reference member function on it, flattens the same scene into the arrays the
oracle (and the C ABI) take -- projections with the cv::Mat arithmetic mirrored in numpy, tests/ref_matcher_lib.py --
and requires identical match indices and counts.  CPU only."""
import numpy as np
import pytest

import ref_matcher_lib as R
from swarmmap_b200 import synth
from swarmmap_b200.matcher import FeatureVector, Frame

pytestmark = pytest.mark.skipif(not R.available(), reason="needs oracle/_ref/liborbmatcher_ref.so, compiled by `make -C oracle ref` "
                                                          "from the reference project's sources, which the repository does not contain")

W, H = 640, 400
K = R.EUROC_K
TH_LOW, TH_HIGH = 50, 100


@pytest.fixture(scope="module")
def scales():
    return R.Scales(1.2, 8)


@pytest.fixture(scope="module")
def frames(oracle):
    seq = synth.make_sequence(4, W, H, 77)
    ex = oracle.Extractor(600, 1.2, 8, 20, 7)
    sf = oracle.scale_tables(1.2, 8)[0]
    return [Frame.from_keypoints(*ex(img), W, H, sf) for img in seq]


def random_frame(rng, n, bits=None, bounds=(0.0, 0.0, float(W), float(H)), cluster=False):
    """Synthetic frame: tie-heavy when `bits` is small (descriptors differ in few bits), clustered positions."""
    if cluster:
        c = rng.uniform([40, 40], [W - 40, H - 40], (12, 2))
        xy = c[rng.integers(0, 12, n)] + rng.normal(0, 9, (n, 2))
    else:
        xy = rng.uniform([bounds[0] - 5, bounds[1] - 5], [bounds[2] + 5, bounds[3] + 5], (n, 2))
    octave = rng.integers(0, 8, n)
    angle = rng.uniform(0, 360, n)
    if bits is None:
        desc = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    else:
        base = rng.integers(0, 256, (1, 32), dtype=np.uint8)
        flip = np.zeros((n, 256), np.uint8)
        for i in range(n):
            flip[i, rng.integers(0, 256, bits)] = 1
        desc = base ^ np.packbits(flip, axis=1)
    return Frame(xy[:, 0], xy[:, 1], octave, angle, desc, bounds)


# ------------------------------------------------------------------------------------------------ primitives

def test_cv_shim_numerics_match_cv2():
    """The cv::Mat stand-in's accumulation rules (oracle/ref_shim_matcher/opencv2/core/core.hpp) against cv2 4.13."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(5)
    for _ in range(3000):
        Rm = rng.standard_normal((3, 3)).astype(np.float32)
        x = (rng.standard_normal(3) * 5).astype(np.float32)
        t = rng.standard_normal(3).astype(np.float32)
        assert np.array_equal(cv2.gemm(Rm, x.reshape(3, 1), 1.0, t.reshape(3, 1), 1.0).ravel(), R.gemm_small(Rm, x, t))
        assert np.array_equal(cv2.gemm(Rm, t.reshape(3, 1), -1.0, None, 0.0, flags=cv2.GEMM_1_T).ravel(),
                              R.gemm_t(Rm, t, -1.0))
        assert np.float32(cv2.norm(x.reshape(3, 1))) == R.norm3(x)


def test_descriptor_distance(oracle):
    rng = np.random.default_rng(1)
    a = rng.integers(0, 256, (500, 32), dtype=np.uint8)
    b = rng.integers(0, 256, (500, 32), dtype=np.uint8)
    b[:50] = a[:50]
    b[50:100] = ~a[50:100]
    for i in range(500):
        assert R.descriptor_distance(a[i], b[i]) == oracle.hamming256(a[i], b[i])


def test_three_maxima_vs_oracle_rule(oracle, frames, scales):
    """ComputeThreeMaxima (:1475-1506) feeds every orientation check; exercised through the matchers below, and here
    directly on tie-heavy histograms against a literal reading."""
    rng = np.random.default_rng(2)
    for _ in range(500):
        sizes = rng.integers(0, 6, 30) * rng.integers(0, 2, 30)
        got = R.three_maxima(sizes)
        m = [0, 0, 0]; ind = [-1, -1, -1]
        for i, s in enumerate(sizes):
            if s > m[0]:
                m = [s, m[0], m[1]]; ind = [i, ind[0], ind[1]]
            elif s > m[1]:
                m = [m[0], s, m[1]]; ind = [ind[0], i, ind[1]]
            elif s > m[2]:
                m[2] = s; ind[2] = i
        if m[1] < np.float32(0.1) * np.float32(m[0]):
            ind[1] = ind[2] = -1
        elif m[2] < np.float32(0.1) * np.float32(m[0]):
            ind[2] = -1
        assert list(got) == ind


@pytest.mark.parametrize("bounds", [(0.0, 0.0, 640.0, 400.0), (-31.4, -17.9, 671.2, 423.3)])
def test_grid_and_features_in_area(oracle, scales, bounds):
    """Frame::AssignFeaturesToGrid / PosInGrid / GetFeaturesInArea: cells, order inside cells, window enumeration
    order and the level-filter rule of Frame.cc:398."""
    import ctypes as C
    rng = np.random.default_rng(3)
    f = random_frame(rng, 900, bounds=bounds)
    rf, keep = R.frame(f, scales)
    rs, ri = R.grid_csr(rf)
    os_, oi = oracle.grid_csr(f)
    assert np.array_equal(rs, os_) and np.array_equal(ri, oi)
    fr, k2 = oracle.make_frame(f.x, f.y, f.octave, f.angle, f.desc, f.bounds)
    g = oracle.lib().orc_grid_build(C.byref(fr))
    out = np.zeros(f.N, np.int32)
    levels = [(-1, -1), (0, 0), (0, -1), (2, -1), (-1, 0), (1, 3), (3, 1), (7, 7), (-1, 2)]
    try:
        for q in range(400):
            x = float(np.float32(rng.uniform(bounds[0] - 60, bounds[2] + 60)))
            y = float(np.float32(rng.uniform(bounds[1] - 60, bounds[3] + 60)))
            r = float(np.float32(rng.choice([0.5, 3.0, 15.0, 40.0, 100.0, 900.0])))
            lo, hi = levels[q % len(levels)]
            ref = R.features_in_area(rf, x, y, r, lo, hi)
            fn = oracle.lib().orc_grid_query
            fn.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_int]
            n = fn(g, C.byref(fr), x, y, r, lo, hi, out.ctypes.data_as(C.c_void_p), f.N)
            assert np.array_equal(ref, out[:n]), (q, x, y, r, lo, hi)
    finally:
        oracle.lib().orc_grid_destroy(g)


def test_keyframe_features_in_area_equals_frame_without_levels(scales):
    """KeyFrame::GetFeaturesInArea (KeyFrame.cc:779-814) = Frame's with the level filter off (integer bounds)."""
    rng = np.random.default_rng(4)
    f = random_frame(rng, 700)
    rf, keep = R.frame(f, scales)
    for q in range(200):
        x, y = float(np.float32(rng.uniform(-30, W + 30))), float(np.float32(rng.uniform(-30, H + 30)))
        r = float(np.float32(rng.choice([2.0, 12.0, 60.0])))
        assert np.array_equal(R.kf_features_in_area(rf, x, y, r), R.features_in_area(rf, x, y, r))


# ------------------------------------------------------------------------------------------------ M1

@pytest.mark.parametrize("ratio,ori", [(0.9, True), (0.9, False), (0.6, True)])
def test_search_for_initialization(oracle, frames, scales, ratio, ori):
    """Three frames with vbPrevMatched carried across calls (Tracking.cc:470-472): steal rule, `<=` / `<` asymmetry,
    orientation pruning, prev update."""
    f0 = frames[0]
    prev_ref = np.stack([f0.x, f0.y], 1).astype(np.float32)
    prev_orc = prev_ref.copy()
    rf0, k0 = R.frame(f0, scales)
    total = 0
    for k in (1, 2, 3):
        rfk, kk = R.frame(frames[k], scales)
        n_ref, m_ref, prev_ref = R.search_for_initialization(rf0, rfk, prev_ref, 100, ratio, ori)
        n_orc, m_orc, prev_orc = oracle.search_for_initialization(f0, frames[k], prev_orc, 100, ratio, ori)
        assert n_ref == n_orc and np.array_equal(m_ref, m_orc) and np.array_equal(prev_ref, prev_orc)
        total += n_ref
    assert total > 100


def test_search_for_initialization_tie_heavy(oracle, scales):
    rng = np.random.default_rng(6)
    for bits in (3, 8, 20):
        a = random_frame(rng, 500, bits=bits, cluster=True)
        b = random_frame(rng, 500, bits=bits, cluster=True)
        a.octave[:] = rng.integers(0, 2, a.N)
        b.octave[:] = rng.integers(0, 2, b.N)
        prev = np.stack([a.x, a.y], 1).astype(np.float32)
        ra, ka = R.frame(a, scales)
        rb, kb = R.frame(b, scales)
        for ratio in (0.9, 1.5):  # > 1: ties at the minimum still pass `best < second * ratio`
            n_ref, m_ref, p_ref = R.search_for_initialization(ra, rb, prev, 60, ratio, True)
            n_orc, m_orc, p_orc = oracle.search_for_initialization(a, b, prev, 60, ratio, True)
            assert n_ref == n_orc and np.array_equal(m_ref, m_orc) and np.array_equal(p_ref, p_orc)


# ------------------------------------------------------------------------------------------------ scenes with poses

def small_pose(rng, rot=0.01, trans=0.03):
    w = rng.normal(0, rot, 3)
    th = np.linalg.norm(w)
    k = w / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    Rm = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx
    T = np.eye(4, dtype=np.float32)
    T[:3, :3] = Rm.astype(np.float32)
    T[:3, 3] = rng.normal(0, trans, 3).astype(np.float32)
    return T


def backproject(f, depth):
    fx, fy, cx, cy = K
    return np.stack([(f.x - cx) / fx * depth, (f.y - cy) / fy * depth, depth], 1).astype(np.float32)


def to_camera(T, pw):
    return np.stack([R.gemm_small(T[:3, :3], p, T[:3, 3]) for p in pw])


def camera_centre(T):
    return R.gemm_t(T[:3, :3], T[:3, 3], -1.0)


@pytest.mark.parametrize("th,ori", [(15.0, True), (30.0, True), (15.0, False)])
def test_search_by_projection_last_frame(oracle, frames, scales, th, ori):
    """SearchByProjection(cur, last, th, bMono = true), :1223-1354 (Tracking.cc:731,736)."""
    rng = np.random.default_rng(8)
    last, cur = frames[0], frames[1]
    n = last.N
    pw = backproject(last, rng.uniform(2, 6, n).astype(np.float32))
    has_mp = rng.random(n) < 0.85
    mp_index = np.where(has_mp, np.arange(n), -1).astype(np.int32)
    outlier = (rng.random(n) < 0.05).astype(np.uint8)
    nobs = rng.integers(0, 3, n).astype(np.int32)
    # a few points behind the camera / outside the image
    pw[rng.choice(n, 10, replace=False), 2] *= -1
    pw[rng.choice(n, 10, replace=False), 0] += 40
    # current frame already holds some points (with and without observations): extra points at the table's end
    n_extra = 60
    extra_slots = rng.choice(cur.N, n_extra, replace=False)
    cur_mp = np.full(cur.N, -1, np.int32)
    cur_mp[extra_slots] = n + np.arange(n_extra)
    nobs_all = np.concatenate([nobs, rng.integers(0, 2, n_extra)]).astype(np.int32)
    pos_all = np.concatenate([pw, np.zeros((n_extra, 3), np.float32)])
    desc_all = np.concatenate([last.desc, np.zeros((n_extra, 32), np.uint8)])
    T = small_pose(rng)
    rp, kp = R.points(pos_all, desc_all, nobs=nobs_all)
    rl, kl = R.frame(last, scales, mp_index=mp_index, outlier=outlier)
    rc, kc = R.frame(cur, scales, Tcw=T, mp_index=cur_mp)
    n_ref, asg_ref = R.search_by_projection_last(rc, rl, rp, th, 0.9, ori)

    pc = to_camera(T, pw)
    u = np.zeros(n, np.float32); v = np.zeros(n, np.float32); valid = np.zeros(n, np.uint8)
    for i in range(n):
        if not has_mp[i] or outlier[i]:
            continue
        ui, vi, invz = R.project(K, pc[i])
        if invz < 0 or ui < 0 or ui > W or vi < 0 or vi > H:
            continue
        u[i], v[i], valid[i] = ui, vi, 1
    radius = (np.float32(th) * scales.sf[last.octave]).astype(np.float32)
    blocked = np.zeros(cur.N, np.uint8)
    blocked[extra_slots] = nobs_all[n:] > 0
    sentinel = np.full(cur.N, -3, np.int32)
    n_orc, asg = oracle.match_window(cur, last.desc, u, v, radius, last.octave - 1, last.octave + 1, valid,
                                     (nobs > 0).astype(np.uint8), TH_HIGH, 0, 0.9, ori, angle=last.angle,
                                     tgt_blocked=blocked, assignment=sentinel)
    expect = np.where(asg == -3, cur_mp, np.where(asg >= 0, mp_index[np.maximum(asg, 0)], -1))
    assert n_ref == n_orc and n_ref > 100
    assert np.array_equal(asg_ref, expect)


@pytest.mark.parametrize("th,ratio", [(1.0, 0.8), (3.0, 0.8), (5.0, 0.95)])
def test_search_by_projection_map_points(oracle, frames, scales, th, ratio):
    """SearchByProjection(F, vpMapPoints, th), :44-121 (Tracking.cc:998-1005): same-level ratio rule, later points
    overwrite, slots holding a point with observations are unavailable."""
    rng = np.random.default_rng(9)
    F, src = frames[2], frames[1]
    m = src.N
    track = dict(in_view=(rng.random(m) < 0.9).astype(np.uint8),
                 proj_x=(src.x + rng.normal(0, 2.0, m)).astype(np.float32),
                 proj_y=(src.y + rng.normal(0, 2.0, m)).astype(np.float32),
                 view_cos=rng.choice([0.9, 0.9985, 0.998, 1.0], m).astype(np.float32),
                 level=np.clip(src.octave + rng.integers(-1, 2, m), 0, 7).astype(np.int32))
    nobs = rng.integers(0, 3, m).astype(np.int32)
    bad = (rng.random(m) < 0.05).astype(np.uint8)
    n_extra = 40
    slots = rng.choice(F.N, n_extra, replace=False)
    f_mp = np.full(F.N, -1, np.int32)
    f_mp[slots] = m + np.arange(n_extra)
    nobs_all = np.concatenate([nobs, rng.integers(0, 2, n_extra)]).astype(np.int32)
    tr_all = {k: np.concatenate([a, np.zeros(n_extra, a.dtype)]) for k, a in track.items()}
    rp, kp = R.points(np.zeros((m + n_extra, 3), np.float32), np.concatenate([src.desc, np.zeros((n_extra, 32), np.uint8)]),
                      nobs=nobs_all, bad=np.concatenate([bad, np.zeros(n_extra, np.uint8)]), track=tr_all)
    rf, kf = R.frame(F, scales, mp_index=f_mp)
    order = rng.permutation(m).astype(np.int32)
    n_ref, asg_ref = R.search_by_projection_points(rf, rp, order, th, ratio)

    r = np.where(track["view_cos"].astype(np.float64) > 0.998, np.float32(2.5), np.float32(4.0)).astype(np.float32)  # float vs double literal
    if th != 1.0:
        r = (r * np.float32(th)).astype(np.float32)
    lvl = track["level"]
    radius = (r * scales.sf[lvl]).astype(np.float32)
    valid = (track["in_view"] != 0) & (bad == 0)
    blocked = np.zeros(F.N, np.uint8)
    blocked[slots] = nobs_all[m:] > 0
    o = order
    n_orc, asg = oracle.match_window(F, src.desc[o], track["proj_x"][o], track["proj_y"][o], radius[o], lvl[o] - 1,
                                     lvl[o], valid[o].astype(np.uint8), (nobs[o] > 0).astype(np.uint8), TH_HIGH, 1,
                                     ratio, False, tgt_blocked=blocked, assignment=np.full(F.N, -3, np.int32))
    expect = np.where(asg == -3, f_mp, np.where(asg >= 0, o[np.maximum(asg, 0)], -1))
    assert n_ref == n_orc and n_ref > 50
    assert np.array_equal(asg_ref, expect)


def test_is_in_frustum_feeds_the_same_fields(frames, scales):
    """Frame::isInFrustum (Frame.cc:316-375) produces the tracking fields the previous test takes as given; the numpy
    mirror of its arithmetic (what host/ORBmatcher.h's callers hold) reproduces them bit for bit."""
    rng = np.random.default_rng(10)
    f = frames[0]
    n = f.N
    pw = backproject(f, rng.uniform(1.5, 8, n).astype(np.float32))
    normal = np.tile(np.array([0, 0, 1], np.float32), (n, 1)) + rng.normal(0, 0.3, (n, 3)).astype(np.float32)
    maxd = rng.uniform(3, 12, n).astype(np.float32)
    mind = (maxd / np.float32(3.5)).astype(np.float32)
    T = small_pose(rng, 0.03, 0.1)
    rp, kp = R.points(pw, f.desc, normal=normal, min_dist=mind, max_dist=maxd)
    rf, kf = R.frame(f, scales, Tcw=T)
    got = R.is_in_frustum(rf, rp, 0.5)
    Ow = camera_centre(T)
    pc = to_camera(T, pw)
    fx, fy, cx, cy = [np.float32(k) for k in K]
    seen = 0
    for i in range(n):
        ok = pc[i, 2] >= 0
        if ok:
            invz = np.float32(np.float32(1.0) / pc[i, 2])
            u = np.float32(np.float32(np.float32(fx * pc[i, 0]) * invz) + cx)
            v = np.float32(np.float32(np.float32(fy * pc[i, 1]) * invz) + cy)
            ok = not (u < 0 or u > W or v < 0 or v > H)
        if ok:
            PO = (pw[i] - Ow).astype(np.float32)
            dist = R.norm3(PO)
            ok = not (dist < np.float32(0.8) * mind[i] or dist > np.float32(1.2) * maxd[i])
        if ok:
            dot = np.float64(PO[0]) * np.float64(normal[i, 0]) + np.float64(PO[1]) * np.float64(normal[i, 1]) \
                + np.float64(PO[2]) * np.float64(normal[i, 2])
            vc = np.float32(dot / np.float64(dist))
            ok = not (vc < np.float32(0.5))
        assert bool(got["in_view"][i]) == bool(ok), i
        if ok:
            seen += 1
            assert got["proj_x"][i] == u and got["proj_y"][i] == v and got["view_cos"][i] == vc
            assert got["level"][i] == R.predict_scale([maxd[i]], [dist], scales.log_sf, 8)[0]
    assert seen > 100


# ------------------------------------------------------------------------------------------------ M4

def bow_nodes(rng, f, n_nodes=90, drop=0.03):
    node = (f.desc[:, 0].astype(np.int64) * 7 + f.desc[:, 5]) % n_nodes + 3 * (np.arange(f.N) % 2)
    node[rng.random(f.N) < drop] = -1  # features whose word has weight 0 are in no node
    return FeatureVector(node)


@pytest.mark.parametrize("ratio,ori", [(0.7, True), (0.75, True), (0.9, False)])
def test_search_by_bow_keyframe_frame(oracle, frames, scales, ratio, ori):
    """SearchByBoW(KeyFrame*, Frame&, ...), :150-262 (Tracking.cc:626,1171)."""
    rng = np.random.default_rng(11)
    kf, F = frames[0], frames[1]
    fv1, fv2 = bow_nodes(rng, kf), bow_nodes(rng, F)
    has = rng.random(kf.N) < 0.8
    mp = np.where(has, np.arange(kf.N), -1).astype(np.int32)
    bad = (rng.random(kf.N) < 0.05).astype(np.uint8)
    rp, kp = R.points(np.zeros((kf.N, 3), np.float32), kf.desc, bad=bad)
    rk, kk = R.frame(kf, scales, mp_index=mp, fv=fv1)
    rf, kf_ = R.frame(F, scales, fv=fv2)
    n_ref, out_ref = R.search_by_bow_kf_f(rk, rf, rp, ratio, ori)
    n_orc, out = oracle.search_by_bow(kf, fv1, (has & (bad == 0)).astype(np.uint8), F, fv2, None, 0, ratio, ori)
    assert n_ref == n_orc and n_ref > 30
    assert np.array_equal(out_ref, out)  # point index == KF keypoint index in this scene


@pytest.mark.parametrize("ratio,ori", [(0.75, True), (0.8, False)])
def test_search_by_bow_keyframe_keyframe(oracle, frames, scales, ratio, ori):
    """SearchByBoW(KeyFrame*, KeyFrame*, ...), :481-597 (LoopClosing.cc:242, AgentMediator.cc:252): `< TH_LOW`."""
    rng = np.random.default_rng(12)
    k1, k2 = frames[1], frames[2]
    fv1, fv2 = bow_nodes(rng, k1), bow_nodes(rng, k2)
    has1, has2 = rng.random(k1.N) < 0.8, rng.random(k2.N) < 0.8
    mp1 = np.where(has1, np.arange(k1.N), -1).astype(np.int32)
    mp2 = np.where(has2, k1.N + np.arange(k2.N), -1).astype(np.int32)
    bad = (rng.random(k1.N + k2.N) < 0.05).astype(np.uint8)
    rp, kp = R.points(np.zeros((k1.N + k2.N, 3), np.float32), np.concatenate([k1.desc, k2.desc]), bad=bad)
    r1, a1 = R.frame(k1, scales, mp_index=mp1, fv=fv1)
    r2, a2 = R.frame(k2, scales, mp_index=mp2, fv=fv2)
    n_ref, out_ref = R.search_by_bow_kf_kf(r1, r2, rp, ratio, ori)
    v1 = (has1 & (bad[:k1.N] == 0)).astype(np.uint8)
    v2 = (has2 & (bad[k1.N:] == 0)).astype(np.uint8)
    n_orc, out = oracle.search_by_bow(k1, fv1, v1, k2, fv2, v2, 1, ratio, ori)
    assert n_ref == n_orc and n_ref > 20
    assert np.array_equal(out_ref, np.where(out >= 0, k1.N + out, -1))


def test_search_by_bow_tie_heavy(oracle, scales):
    rng = np.random.default_rng(13)
    for bits in (4, 12, 30):
        a = random_frame(rng, 400, bits=bits)
        b = random_frame(rng, 400, bits=bits)
        fv1, fv2 = bow_nodes(rng, a, 25), bow_nodes(rng, b, 25)
        rp, kp = R.points(np.zeros((a.N, 3), np.float32), a.desc)
        ra, ka = R.frame(a, scales, mp_index=np.arange(a.N, dtype=np.int32), fv=fv1)
        rb, kb = R.frame(b, scales, fv=fv2)
        for ratio in (0.7, 1.2):
            n_ref, out_ref = R.search_by_bow_kf_f(ra, rb, rp, ratio, True)
            n_orc, out = oracle.search_by_bow(a, fv1, np.ones(a.N, np.uint8), b, fv2, None, 0, ratio, True)
            assert n_ref == n_orc and np.array_equal(out_ref, out)


# ------------------------------------------------------------------------------------------------ M5

def test_search_by_projection_relocalisation(oracle, frames, scales):
    """SearchByProjection(cur, pKF, sAlreadyFound, th, ORBdist, bGlobal), :1356-1473 (Tracking.cc:1235,1248)."""
    rng = np.random.default_rng(14)
    kf, cur = frames[0], frames[1]
    n = kf.N
    depth = rng.uniform(2, 6, n).astype(np.float32)
    pw = backproject(kf, depth)
    has = rng.random(n) < 0.85
    mp = np.where(has, np.arange(n), -1).astype(np.int32)
    bad = (rng.random(n) < 0.05).astype(np.uint8)
    maxd = (depth * rng.uniform(1.0, 2.5, n)).astype(np.float32)
    mind = (maxd / np.float32(3.58)).astype(np.float32)
    found = rng.choice(n, 30, replace=False).astype(np.int32)
    cur_mp = np.full(cur.N, -1, np.int32)
    slots = rng.choice(cur.N, 50, replace=False)
    cur_mp[slots] = found[rng.integers(0, 30, 50)]
    T = small_pose(rng)
    rp, kp = R.points(pw, kf.desc, bad=bad, min_dist=mind, max_dist=maxd)
    rk, kk = R.frame(kf, scales, mp_index=mp)
    rc, kc = R.frame(cur, scales, Tcw=T, mp_index=cur_mp)
    for th, orb_dist in ((10.0, 100), (3.0, 64)):
        n_ref, asg_ref = R.search_by_projection_reloc(rc, rk, rp, found, th, orb_dist, 0.9, True)
        Ow = camera_centre(T)
        pc = to_camera(T, pw)
        u = np.zeros(n, np.float32); v = np.zeros(n, np.float32); valid = np.zeros(n, np.uint8)
        dist = np.ones(n, np.float32)
        for i in range(n):
            if not has[i] or bad[i] or i in found:
                continue
            ui, vi, _ = R.project(K, pc[i])
            if ui < 0 or ui > W or vi < 0 or vi > H:
                continue
            d = R.norm3((pw[i] - Ow).astype(np.float32))
            if d < np.float32(0.8) * mind[i] or d > np.float32(1.2) * maxd[i]:
                continue
            u[i], v[i], valid[i], dist[i] = ui, vi, 1, d
        pred = R.predict_scale(maxd, dist, scales.log_sf, 8)
        radius = (np.float32(th) * scales.sf[pred]).astype(np.float32)
        n_orc, asg = oracle.match_window(cur, kf.desc, u, v, radius, pred - 1, pred + 1, valid, np.ones(n, np.uint8),
                                         orb_dist, 0, 0.9, True, angle=kf.angle,
                                         tgt_blocked=(cur_mp >= 0).astype(np.uint8),
                                         assignment=np.full(cur.N, -3, np.int32))
        expect = np.where(asg == -3, cur_mp, asg)
        assert n_ref == n_orc and n_ref > 50
        assert np.array_equal(asg_ref, expect)


def sim3_decompose(S):
    """ORBmatcher.cc:272-276 with the cv::Mat rules of the header comment in oracle/ref_shim_matcher."""
    sR = S[:3, :3].astype(np.float32)
    dot = sum(np.float64(sR[0, c]) * np.float64(sR[0, c]) for c in range(3))
    scw = np.float32(np.sqrt(dot))  # sqrt(double) -> const float
    inv = np.float32(1.0 / np.float64(scw))
    Rcw = (sR * inv).astype(np.float32)
    tcw = (S[:3, 3].astype(np.float32) * inv).astype(np.float32)
    Ow = R.gemm_t(Rcw, tcw, -1.0)
    return Rcw, tcw, Ow


def project_xy(K, pc, one_is_int):
    """x = xc * invz; u = fx * x + cx (:299-304, :781-786, :940-945)."""
    fx, fy, cx, cy = [np.float32(k) for k in K]
    invz = np.float32(np.float32(1.0) / pc[2]) if one_is_int else np.float32(1.0 / np.float64(pc[2]))
    x = np.float32(pc[0] * invz); y = np.float32(pc[1] * invz)
    return np.float32(np.float32(fx * x) + cx), np.float32(np.float32(fy * y) + cy)


def visible_checks(pw, pc, Ow, normal, mind, maxd, one_is_int, neg_depth_cmp=np.float32(0.0)):
    """The caller-side gates shared by the Sim3 projection / Fuse overloads; returns (valid, u, v, dist)."""
    n = len(pw)
    u = np.zeros(n, np.float32); v = np.zeros(n, np.float32); valid = np.zeros(n, np.uint8); dist = np.ones(n, np.float32)
    for i in range(n):
        if pc[i, 2] < 0:
            continue
        ui, vi = project_xy(K, pc[i], one_is_int)
        if not (ui >= 0 and ui < W and vi >= 0 and vi < H):  # KeyFrame::IsInImage
            continue
        PO = (pw[i] - Ow).astype(np.float32)
        d = R.norm3(PO)
        if d < np.float32(0.8) * mind[i] or d > np.float32(1.2) * maxd[i]:
            continue
        dot = np.float64(PO[0]) * np.float64(normal[i, 0]) + np.float64(PO[1]) * np.float64(normal[i, 1]) \
            + np.float64(PO[2]) * np.float64(normal[i, 2])
        if dot < 0.5 * np.float64(d):
            continue
        u[i], v[i], valid[i], dist[i] = ui, vi, 1, d
    return valid, u, v, dist


def sim3_scene(rng, kf, scale=1.0, rot=0.01, trans=0.03):
    n = kf.N
    depth = rng.uniform(2, 6, n).astype(np.float32)
    pw = backproject(kf, depth)
    normal = np.tile(np.array([0, 0, 1], np.float32), (n, 1)) + rng.normal(0, 0.35, (n, 3)).astype(np.float32)
    maxd = (depth * rng.uniform(1.0, 2.5, n)).astype(np.float32)
    mind = (maxd / np.float32(3.58)).astype(np.float32)
    T = small_pose(rng, rot, trans)
    S = T.copy()
    S[:3, :] *= np.float32(scale)
    return pw, normal, mind, maxd, S


@pytest.mark.parametrize("scale", [1.0, 1.37])
def test_search_by_projection_sim3(oracle, frames, scales, scale):
    """SearchByProjection(pKF, Scw, vpPoints, vpMatched, th), :264-373 (LoopClosing.cc:347)."""
    rng = np.random.default_rng(15)
    kf, src = frames[1], frames[0]
    pw, normal, mind, maxd, S = sim3_scene(rng, src, scale)
    pw = (pw / np.float32(scale)).astype(np.float32)
    m = src.N
    bad = (rng.random(m) < 0.05).astype(np.uint8)
    matched = np.full(kf.N, -1, np.int32)
    slots = rng.choice(kf.N, 40, replace=False)
    matched[slots] = rng.choice(m, 40, replace=False)
    rp, kp = R.points(pw, src.desc, bad=bad, normal=normal, min_dist=mind, max_dist=maxd)
    rk, kk = R.frame(kf, scales)
    order = rng.permutation(m).astype(np.int32)
    n_ref, m_ref = R.search_by_projection_sim3(rk, S, rp, order, matched, 10)
    Rcw, tcw, Ow = sim3_decompose(S)
    pc = np.stack([R.gemm_small(Rcw, p, tcw) for p in pw])
    valid, u, v, dist = visible_checks(pw, pc, Ow, normal, mind, maxd, True)
    valid &= (bad == 0)
    valid[matched[matched >= 0]] = 0
    pred = R.predict_scale(maxd, dist, scales.log_sf, 8)
    radius = (np.float32(10) * scales.sf[pred]).astype(np.float32)
    o = order
    n_orc, asg = oracle.match_window(kf, src.desc[o], u[o], v[o], radius[o], pred[o] - 1, pred[o], valid[o],
                                     np.ones(m, np.uint8), TH_LOW, 0, 0.75, False,
                                     tgt_blocked=(matched >= 0).astype(np.uint8), assignment=np.full(kf.N, -3, np.int32))
    expect = np.where(asg == -3, matched, np.where(asg >= 0, o[np.maximum(asg, 0)], -1))
    assert n_ref == n_orc and n_ref > 30
    assert np.array_equal(m_ref, expect)


# ------------------------------------------------------------------------------------------------ (f)3 rows

def test_search_for_triangulation(oracle, frames, scales):
    """SearchForTriangulation, :599-749 with CheckDistEpipolarLine :131-148 (LocalMapping)."""
    rng = np.random.default_rng(16)
    k1, k2 = frames[0], frames[1]
    # coarse nodes (top bits of one descriptor byte) so that corresponding features usually share a node
    fv1, fv2 = FeatureVector(k1.desc[:, 3] >> 4), FeatureVector(k2.desc[:, 3] >> 4)
    mp1 = np.where(rng.random(k1.N) < 0.3, np.arange(k1.N), -1).astype(np.int32)
    mp2 = np.where(rng.random(k2.N) < 0.3, k1.N + np.arange(k2.N), -1).astype(np.int32)
    T1, T2 = small_pose(rng, 0.02, 0.2), small_pose(rng, 0.02, 0.2)
    rp, kp = R.points(np.zeros((k1.N + k2.N, 3), np.float32), np.concatenate([k1.desc, k2.desc]))
    r1, a1 = R.frame(k1, scales, Tcw=T1, mp_index=mp1, fv=fv1)
    r2, a2 = R.frame(k2, scales, Tcw=T2, mp_index=mp2, fv=fv2)
    # pure sideways camera motion: epipolar lines are the rows (distance = |y2 - y1|), so the gate 3.84 * sigma2
    # splits the candidates of this slowly moving sequence; a little noise makes every term of the line matter
    F12 = np.array([[0, 0, 0], [0, 0, -1], [0, 1, 0]], np.float32) + rng.normal(0, 2e-5, (3, 3)).astype(np.float32)
    for ori in (True, False):
        n_ref, pairs = R.search_for_triangulation(r1, r2, rp, F12, ori)
        Cw = camera_centre(T1)
        C2 = R.gemm_small(T2[:3, :3], Cw, T2[:3, 3])
        fx, fy, cx, cy = [np.float32(k) for k in K]
        invz = np.float32(np.float32(1.0) / C2[2])
        ex = np.float32(np.float32(np.float32(fx * C2[0]) * invz) + cx)
        ey = np.float32(np.float32(np.float32(fy * C2[1]) * invz) + cy)
        n_orc, m12 = oracle.search_for_triangulation(k1, fv1, (mp1 < 0).astype(np.uint8), k2, fv2,
                                                     (mp2 < 0).astype(np.uint8), F12, ex, ey, scales.sf, scales.sigma2, ori)
        exp = np.stack([np.nonzero(m12 >= 0)[0], m12[m12 >= 0]], 1)
        assert n_ref == n_orc and n_ref > 20
        assert np.array_equal(pairs, exp)


def test_fuse(oracle, frames, scales):
    """Fuse(pKF, vpMapPoints, th), :751-893: search loop through the oracle, bookkeeping replayed in list order."""
    rng = np.random.default_rng(17)
    kf = src = frames[0]  # the points are the keyframe's own features seen from a slightly different pose (~1 px)
    pw, normal, mind, maxd, T = sim3_scene(rng, src, 1.0, 0.001, 0.003)
    m = src.N
    bad = (rng.random(m) < 0.05).astype(np.uint8)
    nobs = rng.integers(1, 6, m + kf.N).astype(np.int32)
    # the keyframe already holds points (table entries m..): some of them bad
    kf_mp = np.where(rng.random(kf.N) < 0.5, m + np.arange(kf.N), -1).astype(np.int32)
    bad_all = np.concatenate([bad, (rng.random(kf.N) < 0.1).astype(np.uint8)])
    rp, kp = R.points(np.concatenate([pw, np.zeros((kf.N, 3), np.float32)]),
                      np.concatenate([src.desc, np.zeros((kf.N, 32), np.uint8)]), nobs=nobs, bad=bad_all,
                      normal=np.concatenate([normal, np.zeros((kf.N, 3), np.float32)]),
                      min_dist=np.concatenate([mind, np.ones(kf.N, np.float32)]),
                      max_dist=np.concatenate([maxd, np.ones(kf.N, np.float32)]))
    rk, kk = R.frame(kf, scales, Tcw=T, mp_index=kf_mp)
    order = rng.permutation(m).astype(np.int32)
    order[rng.choice(m, 8, replace=False)] = -1  # NULL entries (:769-770)
    n_ref, asg_ref, rep_ref = R.fuse(rk, rp, order, 3.0)

    Ow = camera_centre(T)
    pc = to_camera(T, pw)
    valid, u, v, dist = visible_checks(pw, pc, Ow, normal, mind, maxd, True)
    valid &= (bad == 0)
    pred = R.predict_scale(maxd, dist, scales.log_sf, 8)
    radius = (np.float32(3.0) * scales.sf[pred]).astype(np.float32)
    bi, bd = oracle.window_best(kf, src.desc, u, v, radius, pred, valid, scales.inv_sigma2, 5.99)
    asg = kf_mp.copy(); rep = np.full(m + kf.N, -1, np.int32); isbad = bad_all.copy(); nfused = 0
    in_kf = set()
    for p in order:
        if p < 0 or isbad[p] or p in in_kf or not valid[p]:
            continue
        if bi[p] >= 0 and bd[p] <= TH_LOW:
            j = bi[p]
            q = asg[j]
            if q >= 0:
                if not isbad[q]:
                    if nobs[q] > nobs[p]:
                        isbad[p] = 1; rep[p] = q
                    else:
                        isbad[q] = 1; rep[q] = p
            else:
                asg[j] = p; in_kf.add(p); nobs[p] += 1  # AddObservation
            nfused += 1
    assert n_ref == nfused and nfused > 30
    assert np.array_equal(asg_ref, asg) and np.array_equal(rep_ref, rep)


@pytest.mark.parametrize("scale", [1.0, 0.83])
def test_fuse_sim3(oracle, frames, scales, scale):
    """Fuse(pKF, Scw, vpPoints, th, vpReplacePoint), :895-1009."""
    rng = np.random.default_rng(18)
    kf = src = frames[1]
    pw, normal, mind, maxd, S = sim3_scene(rng, src, scale, 0.002, 0.006)
    pw = (pw / np.float32(scale)).astype(np.float32)
    m = src.N
    bad = (rng.random(m) < 0.05).astype(np.uint8)
    kf_mp = np.where(rng.random(kf.N) < 0.5, m + np.arange(kf.N), -1).astype(np.int32)
    bad_all = np.concatenate([bad, (rng.random(kf.N) < 0.1).astype(np.uint8)])
    rp, kp = R.points(np.concatenate([pw, np.zeros((kf.N, 3), np.float32)]),
                      np.concatenate([src.desc, np.zeros((kf.N, 32), np.uint8)]), bad=bad_all,
                      normal=np.concatenate([normal, np.zeros((kf.N, 3), np.float32)]),
                      min_dist=np.concatenate([mind, np.ones(kf.N, np.float32)]),
                      max_dist=np.concatenate([maxd, np.ones(kf.N, np.float32)]))
    rk, kk = R.frame(kf, scales, mp_index=kf_mp)
    order = rng.permutation(m).astype(np.int32)
    n_ref, asg_ref, rep_ref = R.fuse_sim3(rk, S, rp, order, 4.0)
    Rcw, tcw, Ow = sim3_decompose(S)
    pc = np.stack([R.gemm_small(Rcw, p, tcw) for p in pw])
    valid, u, v, dist = visible_checks(pw, pc, Ow, normal, mind, maxd, False)
    valid &= (bad == 0)
    pred = R.predict_scale(maxd, dist, scales.log_sf, 8)
    radius = (np.float32(4.0) * scales.sf[pred]).astype(np.float32)
    bi, bd = oracle.window_best(kf, src.desc, u, v, radius, pred, valid, scales.inv_sigma2, 0.0)
    asg = kf_mp.copy(); rep = np.full(m, -1, np.int32); nfused = 0
    for k, p in enumerate(order):
        if not valid[p]:
            continue
        if bi[p] >= 0 and bd[p] <= TH_LOW:
            q = asg[bi[p]]
            if q >= 0:
                if not bad_all[q]:
                    rep[k] = q
            else:
                asg[bi[p]] = p
            nfused += 1
    assert n_ref == nfused and nfused > 30
    assert np.array_equal(asg_ref, asg) and np.array_equal(rep_ref, rep)


def test_search_by_sim3(oracle, frames, scales):
    """SearchBySim3, :1011-1221 (LoopClosing.cc:285): two window searches and the mutual-agreement check."""
    rng = np.random.default_rng(19)
    k1 = k2 = frames[0]  # the same features seen from two slightly different poses with independent depths
    n1, n2 = k1.N, k2.N
    T1, T2 = small_pose(rng, 0.002, 0.006), small_pose(rng, 0.002, 0.006)
    d1, d2 = rng.uniform(2, 6, n1).astype(np.float32), rng.uniform(2, 6, n2).astype(np.float32)
    # world points: back-projections in each keyframe's own camera, moved to the world with the inverse pose
    def to_world(T, pc):
        Rt = T[:3, :3].T.astype(np.float64)
        return ((pc.astype(np.float64) - T[:3, 3].astype(np.float64)) @ Rt.T).astype(np.float32)
    pw = np.concatenate([to_world(T1, backproject(k1, d1)), to_world(T2, backproject(k2, d2))])
    has1, has2 = rng.random(n1) < 0.8, rng.random(n2) < 0.8
    mp1 = np.where(has1, np.arange(n1), -1).astype(np.int32)
    mp2 = np.where(has2, n1 + np.arange(n2), -1).astype(np.int32)
    bad = (rng.random(n1 + n2) < 0.04).astype(np.uint8)
    maxd = (np.concatenate([d1, d2]) * rng.uniform(1.0, 2.5, n1 + n2)).astype(np.float32)
    mind = (maxd / np.float32(3.58)).astype(np.float32)
    rp, kp = R.points(pw, np.concatenate([k1.desc, k2.desc]), bad=bad, min_dist=mind, max_dist=maxd)
    r1, a1 = R.frame(k1, scales, Tcw=T1, mp_index=mp1)
    r2, a2 = R.frame(k2, scales, Tcw=T2, mp_index=mp2)
    s12 = np.float32(1.0)
    # relative motion camera 2 -> camera 1
    T12 = (T1.astype(np.float64) @ np.linalg.inv(T2.astype(np.float64))).astype(np.float32)
    R12, t12 = np.ascontiguousarray(T12[:3, :3]), np.ascontiguousarray(T12[:3, 3])
    pre = np.full(n1, -1, np.int32)
    cand = np.nonzero(has2)[0]
    pre_slots = rng.choice(np.nonzero(has1)[0], 25, replace=False)
    pre[pre_slots] = n1 + rng.choice(cand, 25, replace=False)
    n_ref, m_ref = R.search_by_sim3(r1, r2, rp, pre, float(s12), R12, t12, 7.5)

    sR12 = (R12 * np.float32(s12)).astype(np.float32)
    inv_s = np.float32(1.0 / np.float64(s12))
    sR21 = (R12.T * inv_s).astype(np.float32)
    t21 = np.array([np.float32(-1.0 * np.float64(np.float32(np.float32(np.float32(sR21[r, 0] * t12[0]) + np.float32(sR21[r, 1] * t12[1]))
                                                          + np.float32(sR21[r, 2] * t12[2])))) for r in range(3)], np.float32)
    fx, fy, cx, cy = [np.float32(k) for k in K]

    def direction(Ta, sR, tt, idx, maxd_, mind_, tgt):
        n = len(idx)
        u = np.zeros(n, np.float32); v = np.zeros(n, np.float32); valid = np.zeros(n, np.uint8); dist = np.ones(n, np.float32)
        for k, p in enumerate(idx):
            pa = R.gemm_small(Ta[:3, :3], pw[p], Ta[:3, 3])
            pb = R.gemm_small(sR, pa, tt)
            if pb[2] < 0:
                continue
            ui, vi = project_xy(K, pb, False)
            if not (ui >= 0 and ui < W and vi >= 0 and vi < H):
                continue
            d = R.norm3(pb)
            if d < np.float32(0.8) * mind_[k] or d > np.float32(1.2) * maxd_[k]:
                continue
            u[k], v[k], valid[k], dist[k] = ui, vi, 1, d
        pred = R.predict_scale(maxd_, dist, scales.log_sf, 8)
        return u, v, valid, pred

    already1 = pre >= 0
    already2 = np.zeros(n2, bool)
    already2[pre[pre >= 0] - n1] = True
    idx1 = np.arange(n1); idx2 = n1 + np.arange(n2)
    u, v, valid, pred = direction(T1, sR21, t21, idx1, maxd[:n1], mind[:n1], k2)
    valid &= (has1 & ~already1 & (bad[:n1] == 0)).astype(np.uint8)
    b1, dd1 = oracle.window_best(k2, k1.desc, u, v, (np.float32(7.5) * scales.sf[pred]).astype(np.float32), pred, valid,
                                 scales.inv_sigma2, 0.0)
    m1 = np.where((b1 >= 0) & (dd1 <= TH_HIGH), b1, -1)
    u, v, valid, pred = direction(T2, sR12, t12, idx2, maxd[n1:], mind[n1:], k1)
    valid &= (has2 & ~already2 & (bad[n1:] == 0)).astype(np.uint8)
    b2, dd2 = oracle.window_best(k1, k2.desc, u, v, (np.float32(7.5) * scales.sf[pred]).astype(np.float32), pred, valid,
                                 scales.inv_sigma2, 0.0)
    m2 = np.where((b2 >= 0) & (dd2 <= TH_HIGH), b2, -1)
    exp = pre.copy(); found = 0
    for i1 in range(n1):
        if m1[i1] >= 0 and m2[m1[i1]] == i1:
            exp[i1] = mp2[m1[i1]]; found += 1
    assert n_ref == found and found > 30
    assert np.array_equal(m_ref, exp)
