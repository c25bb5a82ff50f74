"""The device's greedy resolve (match.cu resolve_body) against the oracle, bit for bit, where its rules sit on their
edges: every hand-built case of tests/matcher_cases.py, the tie-heavy random generator, and every job of the
benchmark's own batch shapes.  Each input goes through the host-array single call, resident frames and the batched
call, where it sits in slot 0 and in the last slot next to unrelated jobs."""
import numpy as np
import pytest

import matcher_cases
from matcher_cases import random_frame
from swarmmap_b200 import synth

pytestmark = pytest.mark.gpu

CASES = matcher_cases.cases()


def _expect(oracle, case):
    r = case.run_oracle(oracle)
    case.reach(oracle, r)
    return r


def _window_kw(c, tgt):
    return dict(tgt=tgt, desc=c.desc, u=c.u, v=c.v, radius=c.radius, min_level=c.lo, max_level=c.hi, valid=c.valid,
                blocks=c.blocks, th_dist=c.th_dist, ratio_mode=c.ratio_mode, angle=c.angle, tgt_blocked=c.tgt_blocked,
                check_ori=c.check_ori)


def _single(c, resident):
    """One call of the single-problem entry point; resident: the frames are uploaded first.  -> (n, out, prev)."""
    from swarmmap_b200.matcher import ORBmatcher, ResidentFrame
    up = (lambda f: ResidentFrame().upload(f)) if resident else (lambda f: f)
    if c.kind == "init":
        m = ORBmatcher(c.nnratio, c.check_ori)
        prev = c.prev.copy()
        n, m12 = m.SearchForInitialization(up(c.f1), up(c.f2), prev, c.window)
        return n, m12, prev
    if c.kind == "window":
        m = ORBmatcher(c.nnratio, c.check_ori)
        kw = _window_kw(c, up(c.tgt))
        n, asg = m.match_window(**kw)
        return n, asg, None
    m = ORBmatcher(c.nnratio, c.check_ori)
    n, out = m.SearchByBoW(up(c.f1), c.fv1, c.valid1, up(c.f2), c.fv2, c.valid2)
    return n, out, None


def _same(got, exp, what):
    n, out, prev = got
    on, oout, oprev = exp
    assert n == on, (what, n, on)
    np.testing.assert_array_equal(out, oout, err_msg=what)
    if oprev is not None:
        np.testing.assert_array_equal(prev, oprev, err_msg=what)


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_hand_built_single(oracle, swm, case):
    exp = _expect(oracle, case)
    _same(_single(case, False), exp, "host arrays")
    if not (case.kind == "window" and case.tgt.N == 0) and not (case.kind != "window" and case.f2.N == 0):
        _same(_single(case, True), exp, "resident")


# ---- unrelated jobs that share a batch with a case

def _filler(kind, seed, like):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (1, 32), dtype=np.uint8)
    a = random_frame(rng, 300, bits=6, cluster=True, base=base)
    b = random_frame(rng, 300, bits=6, cluster=True, base=base)
    if kind == "init":
        a.octave[:] = rng.integers(0, 2, a.N)
        b.octave[:] = rng.integers(0, 2, b.N)
        return matcher_cases.Case("filler", "init", f1=a, f2=b, prev=np.stack([a.x, a.y], 1).astype(np.float32),
                                  window=like.window, nnratio=like.nnratio, check_ori=like.check_ori)
    if kind == "window":
        m = a.N
        return matcher_cases.Case("filler", "window", tgt=b, desc=a.desc, u=(a.x + rng.normal(0, 3, m)).astype(np.float32),
                                  v=(a.y + rng.normal(0, 3, m)).astype(np.float32), radius=np.full(m, 20, np.float32),
                                  lo=a.octave - 1, hi=a.octave + 1, valid=(rng.random(m) < 0.9).astype(np.uint8),
                                  blocks=(rng.random(m) < 0.7).astype(np.uint8), angle=a.angle,
                                  tgt_blocked=(rng.random(b.N) < 0.1).astype(np.uint8), th_dist=100,
                                  ratio_mode=1 - like.ratio_mode, nnratio=like.nnratio, check_ori=not like.check_ori)
    from swarmmap_b200.matcher import FeatureVector
    node = lambda f: f.desc[:, 3].astype(np.int64) % 7
    mode = like.mode
    return matcher_cases.Case("filler", "bow", f1=a, fv1=FeatureVector(node(a)), valid1=np.ones(a.N, np.uint8), f2=b,
                              fv2=FeatureVector(node(b)), valid2=np.ones(b.N, np.uint8) if mode == 1 else None,
                              mode=mode, nnratio=like.nnratio, check_ori=like.check_ori)


def _batch(cases, resident):
    """One batched call over `cases` (one kind; nnratio and check_ori of the first for Init / BoW)."""
    from swarmmap_b200.matcher import ORBmatcher, ResidentFrame
    cache = {}

    def up(f):
        if not resident:
            return f
        if id(f) not in cache:
            cache[id(f)] = ResidentFrame().upload(f)
        return cache[id(f)]
    c0 = cases[0]
    m = ORBmatcher(c0.nnratio, c0.check_ori)
    if c0.kind == "init":
        prevs = [c.prev.copy() for c in cases]
        got = m.SearchForInitializationBatch([(up(c.f1), up(c.f2), p) for c, p in zip(cases, prevs)], c0.window)
        return [(n, o, p) for (n, o), p in zip(got, prevs)]
    if c0.kind == "window":
        got = m.match_window_batch([_window_kw(c, up(c.tgt)) for c in cases])
        return [(n, o, None) for n, o in got]
    got = m.SearchByBoWBatch([(up(c.f1), c.fv1, c.valid1, up(c.f2), c.fv2, c.valid2) for c in cases])
    return [(n, o, None) for n, o in got]


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_hand_built_batch_first_and_last_slot(oracle, swm, case):
    exp = _expect(oracle, case)
    fill = [_filler(case.kind, s, case) for s in (1, 2, 3)]
    jobs = [case] + fill + [case]
    resident = case.kind == "init" or (case.kind == "window" and case.tgt.N > 0) or (case.kind == "bow" and case.f2.N > 0)
    for res in sorted({False, resident}):
        got = _batch(jobs, res)
        _same(got[0], exp, f"slot 0, resident={res}")
        _same(got[-1], exp, f"last slot, resident={res}")
        for f, g in zip(fill, got[1:-1]):
            _same(g, f.run_oracle(oracle), f"filler, resident={res}")


# ---- the tie-heavy generator at the benchmark's frame shapes

SHAPES = {"euroc": (752, 480, 1000), "kitti": (1241, 376, 4000)}


def _tie_heavy(kind, bits, cluster, shape, seed):
    w, h, n = SHAPES[shape]
    rng = np.random.default_rng(seed)
    bounds = (0.0, 0.0, float(w), float(h))
    base = rng.integers(0, 256, (1, 32), dtype=np.uint8)
    a = random_frame(rng, n, bits=bits, bounds=bounds, cluster=cluster, base=base)
    b = random_frame(rng, n, bits=bits, bounds=bounds, cluster=cluster, base=base)
    like = matcher_cases.Case("like", kind, window=60, nnratio=1.5 if bits == 2 else 0.9, check_ori=True, ratio_mode=0,
                              mode=seed % 2)
    c = _filler(kind, seed, like)
    c.name = f"tie_heavy_{kind}_{bits}_{'cluster' if cluster else 'uniform'}_{shape}"
    if kind == "init":
        a.octave[:] = rng.integers(0, 2, a.N)
        b.octave[:] = rng.integers(0, 2, b.N)
        c.f1, c.f2, c.prev = a, b, np.stack([a.x, a.y], 1).astype(np.float32)
    elif kind == "window":
        m = a.N
        c.tgt, c.desc, c.angle = b, a.desc, a.angle
        c.u = (a.x + rng.normal(0, 3, m)).astype(np.float32)
        c.v = (a.y + rng.normal(0, 3, m)).astype(np.float32)
        c.radius = np.full(m, 25, np.float32)
        c.lo, c.hi = a.octave - 1, a.octave + 1
        c.valid = (rng.random(m) < 0.9).astype(np.uint8)
        c.blocks = (rng.random(m) < 0.7).astype(np.uint8)
        c.tgt_blocked = (rng.random(b.N) < 0.05).astype(np.uint8)
        c.ratio_mode, c.check_ori = seed % 2, seed % 2 == 0
    else:
        from swarmmap_b200.matcher import FeatureVector
        node = lambda f: f.desc[:, 5].astype(np.int64) % 40
        c.f1, c.f2, c.fv1, c.fv2 = a, b, FeatureVector(node(a)), FeatureVector(node(b))
        c.valid1 = (rng.random(a.N) < 0.9).astype(np.uint8)
        c.valid2 = (rng.random(b.N) < 0.9).astype(np.uint8) if c.mode == 1 else None
    return c


TIE = [(k, bits, cl, sh) for k in ("init", "window", "bow") for bits in (2, 4, 8) for cl in (True, False)
       for sh in SHAPES]


@pytest.mark.parametrize("kind,bits,cluster,shape", TIE)
def test_tie_heavy_generator(oracle, swm, kind, bits, cluster, shape):
    c = _tie_heavy(kind, bits, cluster, shape, 1000 + TIE.index((kind, bits, cluster, shape)))
    exp = c.run_oracle(oracle)
    assert exp[0] > 0
    _same(_single(c, False), exp, "host arrays")
    _same(_single(c, True), exp, "resident")
    other = _filler(kind, 7, c)
    got = _batch([c, other, c], True)
    _same(got[0], exp, "slot 0")
    _same(got[2], exp, "last slot")
    _same(got[1], other.run_oracle(oracle), "filler")


# ---- the benchmark's batch shapes: every job of one config34_tracking step and of config2_kitti.init_matching

EUROC_CAM = (458.654, 457.296, 367.215, 248.375, -0.28340811, 0.07395907, 0.00019359, 1.76187114e-05, 0.0)


def test_tracking_step_all_agents(oracle, swm):
    """config34_tracking: 128 agents on 8 sequences (752 x 480, 1000 features), the last timed step.  Map points are
    the previous frame's keypoints (SearchByProjection(cur, last, 15), 0.9, orientation on) and the previous two
    frames' (SearchByProjection(F, points, th 1), ratio_mode 1, 0.8, orientation off), warped by the generator's motion
    plus 1 px noise; SearchByBoW(KF = previous frame, F), 0.7, on FeatureVectors of the device's vocabulary
    transform (k = 10, L = 5 synthetic vocabulary, levelsup 4)."""
    from swarmmap_b200.bow import ORBVocabulary
    from swarmmap_b200.matcher import Camera, FeatureVector, Frame, ORBmatcher, resident_frames_from_extractor
    from swarmmap_b200.orb import ORBextractor
    W, H, S, T, P = 752, 480, 8, 10, 128
    seqs, warps = [], []
    for s in range(S):
        fr, hs = synth.make_sequence(T + 2 + P // S, W, H, 20220406 + s, return_h=True)
        seqs.append(fr)
        warps.append(hs)
    t = T + 1
    frame_of = lambda a, tt: (a % S, a // S + tt)
    ex = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=P)
    sf = ex.GetScaleFactors()
    cam = Camera(*EUROC_CAM)
    bounds = cam.bounds(W, H)
    feats, res = {}, {}
    for tt in (t - 2, t - 1, t):
        k, d, n = ex.extract_batch(np.stack([seqs[frame_of(a, tt)[0]][frame_of(a, tt)[1]] for a in range(P)]))
        feats[tt] = (k.copy(), d.copy(), n.copy())
        if tt >= t - 1:
            res[tt] = resident_frames_from_extractor(ex, P, cam, bounds)

    def host_frame(tt, a):
        k, d, n = feats[tt]
        und = oracle.undistort_points(np.stack([k[a, :n[a]]["x"], k[a, :n[a]]["y"]], 1).astype(np.float32),
                                      np.array(EUROC_CAM, np.float32))
        return Frame(und[:, 0], und[:, 1], k[a, :n[a]]["octave"], k[a, :n[a]]["angle"], d[a, :n[a]],
                     (float(bounds[0]), float(bounds[2]), float(bounds[1]), float(bounds[3])), sf)

    def warp(s, i_from, i_to, x, y):
        A, B2 = np.vstack([warps[s][i_from], [0, 0, 1]]), np.vstack([warps[s][i_to], [0, 0, 1]])
        Mx = np.linalg.inv(B2) @ A
        return ((Mx[0, 0] * x + Mx[0, 1] * y + Mx[0, 2]).astype(np.float32),
                (Mx[1, 0] * x + Mx[1, 1] * y + Mx[1, 2]).astype(np.float32))

    rng = np.random.default_rng(7)
    cur = [host_frame(t, a) for a in range(P)]
    total = 0
    for mode, m in ((0, ORBmatcher(0.9, True)), (1, ORBmatcher(0.8, True))):
        jobs = []
        for a in range(P):
            s, i = frame_of(a, t)
            us, vs, descs, octs, angs = [], [], [], [], []
            for tt in ([t - 1] if mode == 0 else [t - 1, t - 2]):
                k, d, n = feats[tt]
                kk = k[a, :n[a]]
                x, y = warp(s, frame_of(a, tt)[1], i, kk["x"], kk["y"])
                us.append(x + rng.normal(0, 1.0, len(x)).astype(np.float32))
                vs.append(y + rng.normal(0, 1.0, len(x)).astype(np.float32))
                descs.append(d[a, :n[a]])
                octs.append(kk["octave"])
                angs.append(kk["angle"])
            u, v = np.concatenate(us), np.concatenate(vs)
            octv = np.concatenate(octs).astype(np.int32)
            valid = ((u >= bounds[0]) & (u <= bounds[1]) & (v >= bounds[2]) & (v <= bounds[3])).astype(np.uint8)
            th = 15.0 if mode == 0 else 2.5
            jobs.append(dict(tgt=res[t][a], desc=np.concatenate(descs), u=u, v=v,
                             radius=(np.float32(th) * sf[octv]).astype(np.float32), min_level=octv - 1,
                             max_level=octv + 1 if mode == 0 else octv.copy(), valid=valid,
                             blocks=np.ones(len(u), np.uint8), th_dist=100, ratio_mode=mode,
                             angle=np.concatenate(angs).astype(np.float32), check_ori=mode == 0))
        got = m.match_window_batch(jobs)
        for a, (j, (n, asg)) in enumerate(zip(jobs, got)):
            on, oasg = oracle.match_window(cur[a], j["desc"], j["u"], j["v"], j["radius"], j["min_level"],
                                           j["max_level"], j["valid"], j["blocks"], 100, mode, 0.9 if mode == 0 else 0.8,
                                           j["check_ori"], j["angle"])
            assert n == on, (mode, a)
            np.testing.assert_array_equal(asg, oasg, err_msg=f"mode {mode} agent {a}")
            total += n
    # SearchByBoW(KF = previous frame, F): FeatureVectors from the device's transform, equal to the oracle's
    voc = ORBVocabulary(synth.make_vocabulary(10, 5, seed=20220407))
    ov = oracle.Vocabulary(synth.make_vocabulary(10, 5, seed=20220407))
    fvs = {}
    for tt in (t - 1, t):
        k, d, n = feats[tt]
        fvs[tt] = [b.feature_vector() for b in voc.transform_batch(d, n, 4)]
        for a in (0, 77, P - 1):
            o = ov.transform(d[a, :n[a]], 4)
            assert np.array_equal(fvs[tt][a].node_ids, o[2]) and np.array_equal(fvs[tt][a].feats, o[4])
    m7 = ORBmatcher(0.7, True)
    kf = [host_frame(t - 1, a) for a in range(P)]
    got = m7.SearchByBoWBatch([(res[t - 1][a], fvs[t - 1][a], np.ones(kf[a].N, np.uint8), res[t][a], fvs[t][a], None)
                               for a in range(P)])
    for a, (n, out) in enumerate(got):
        on, oout = oracle.search_by_bow(kf[a], fvs[t - 1][a], np.ones(kf[a].N, np.uint8), cur[a], fvs[t][a], None, 0,
                                        0.7, True)
        assert n == on, a
        np.testing.assert_array_equal(out, oout, err_msg=f"bow agent {a}")
        total += n
    assert total > 128 * 300


def test_kitti_init_chains_all(oracle, swm):
    """config2_kitti.init_matching: 89 chains over a 100-frame 1241 x 376 sequence, 4000 features,
    SearchForInitialization(F_0 = frame s, F_k = frame s + k, window 100), k = 1..10, vbPrevMatched carried."""
    from swarmmap_b200.matcher import Frame, ORBmatcher, ResidentFrame
    from swarmmap_b200.orb import ORBextractor
    wk, hk = 1241, 376
    seq = synth.make_sequence(100, wk, hk, 20220405)
    ex = ORBextractor(4000, 1.2, 8, 20, 7, max_batch=100)
    kps, desc, n = ex.extract_batch(seq)
    sf = ex.GetScaleFactors()
    fs = [Frame.from_keypoints(kps[i, :n[i]].copy(), desc[i, :n[i]].copy(), wk, hk, sf) for i in range(100)]
    res = [ResidentFrame().upload(f) for f in fs]
    P, K = 89, 10
    m = ORBmatcher(0.9, True)
    prev = [np.stack([fs[s].x, fs[s].y], 1).astype(np.float32).copy() for s in range(P)]
    oprev = [p.copy() for p in prev]
    for k in range(1, K + 1):
        got = m.SearchForInitializationBatch([(res[s], res[s + k], prev[s]) for s in range(P)], 100)
        for s in range(P):
            on, om12, oprev[s] = oracle.search_for_initialization(fs[s], fs[s + k], oprev[s], 100, 0.9, True)
            assert got[s][0] == on, (s, k)
            np.testing.assert_array_equal(got[s][1], om12, err_msg=f"chain {s} k {k}")
            np.testing.assert_array_equal(prev[s], oprev[s], err_msg=f"prev chain {s} k {k}")
