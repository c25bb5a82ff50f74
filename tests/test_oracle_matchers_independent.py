"""Second, independent (pure numpy / Python) readings of the reference sources for the oracle functions added with
the SURVEY section 8(f) rows, on small seeded inputs: the Fuse / SearchBySim3 search loop incl. a literal
Frame::GetFeaturesInArea (code/src/Frame.cc:377-425), ComputeDistinctiveDescriptors (code/src/MapPoint.cc:361-391) and
SearchForTriangulation's per-row choice (code/src/ORBmatcher.cc:599-749).  The oracle is the checker of the CUDA
path; these tests check the checker."""
import math

import numpy as np
import pytest

import matcher_cases
from swarmmap_b200 import synth

TH_LOW = 50


@pytest.fixture(scope="module")
def two_frames(oracle):
    from swarmmap_b200.matcher import Frame
    seq = synth.make_sequence(2, 640, 400, 99)
    ex = oracle.Extractor(500, 1.2, 8, 20, 7)
    sf = oracle.scale_tables(1.2, 8)[0]
    return [Frame.from_keypoints(*ex(img), 640, 400, sf) for img in seq]


def get_features_in_area(f, grid, x, y, r):
    """Frame.cc:377-425 without level arguments."""
    starts, items = grid
    minx, miny, maxx, maxy = f.bounds
    inv_w = np.float32(64) / np.float32(maxx - minx)
    inv_h = np.float32(48) / np.float32(maxy - miny)
    x, y, r = np.float32(x), np.float32(y), np.float32(r)
    c0 = max(0, int(np.floor((x - np.float32(minx) - r) * inv_w)))
    if c0 >= 64:
        return []
    c1 = min(63, int(np.ceil((x - np.float32(minx) + r) * inv_w)))
    if c1 < 0:
        return []
    r0 = max(0, int(np.floor((y - np.float32(miny) - r) * inv_h)))
    if r0 >= 48:
        return []
    r1 = min(47, int(np.ceil((y - np.float32(miny) + r) * inv_h)))
    if r1 < 0:
        return []
    out = []
    for ix in range(c0, c1 + 1):
        for iy in range(r0, r1 + 1):
            cell = ix * 48 + iy
            for j in items[starts[cell]:starts[cell + 1]]:
                if abs(np.float32(f.x[j]) - x) < r and abs(np.float32(f.y[j]) - y) < r:
                    out.append(int(j))
    return out


def hamming(a, b):
    return int(np.unpackbits(a ^ b).sum())


@pytest.mark.parametrize("chi2", [5.99, 0.0])
def test_window_best_vs_python(oracle, two_frames, chi2):
    src = tgt = two_frames[0]  # projections scatter around the frame's own keypoints: many windows are non-empty
    rng = np.random.default_rng(3)
    sf, _, _, inv_s2 = oracle.scale_tables(1.2, 8)
    m = 150
    u = (src.x[:m] + rng.normal(0, 1.2, m)).astype(np.float32)
    v = (src.y[:m] + rng.normal(0, 1.2, m)).astype(np.float32)
    pred = np.clip(src.octave[:m] + rng.integers(-1, 2, m), 0, 7).astype(np.int32)
    radius = (np.float32(14.0) * sf[pred]).astype(np.float32)
    valid = (rng.random(m) < 0.9).astype(np.uint8)
    bi, bd = oracle.window_best(tgt, src.desc[:m], u, v, radius, pred, valid, inv_s2, chi2)
    grid = oracle.grid_csr(tgt)
    hits = 0
    for i in range(m):
        best_d, best_i = 256, -1
        if valid[i]:
            for j in get_features_in_area(tgt, grid, u[i], v[i], radius[i]):
                lvl = tgt.octave[j]
                if lvl < pred[i] - 1 or lvl > pred[i]:
                    continue
                if chi2 > 0:
                    ex, ey = np.float32(u[i] - tgt.x[j]), np.float32(v[i] - tgt.y[j])
                    e2 = np.float32(np.float32(ex * ex) + np.float32(ey * ey))
                    if float(np.float32(e2 * inv_s2[lvl])) > float(np.float32(chi2)):
                        continue
                d = hamming(src.desc[i], tgt.desc[j])
                if d < best_d:
                    best_d, best_i = d, j
        assert (bi[i], bd[i]) == (best_i, best_d), i
        hits += best_i >= 0
    assert hits > 10


def test_distinctive_descriptors_vs_numpy(oracle):
    rng = np.random.default_rng(5)
    sizes = [1, 2, 3, 4, 9, 10, 0, 25]
    chunks = []
    for n in sizes:
        base = rng.integers(0, 256, 32, dtype=np.uint8)
        bits = np.unpackbits(np.repeat(base[None], n, 0), axis=1) if n else np.zeros((0, 256), np.uint8)
        bits ^= (rng.random(bits.shape) < 0.1).astype(np.uint8)
        chunks.append(np.packbits(bits, axis=1) if n else np.zeros((0, 32), np.uint8))
    desc = np.concatenate(chunks)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    best, med = oracle.distinctive_descriptors(desc, off)
    for p, n in enumerate(sizes):
        if n == 0:
            assert best[p] == -1
            continue
        d = desc[off[p]:off[p + 1]]
        D = np.unpackbits(d[:, None, :] ^ d[None, :, :], axis=2).sum(2)
        meds = [sorted(D[i])[int(0.5 * (n - 1))] for i in range(n)]
        assert med[p] == min(meds) and best[p] == int(np.argmin(meds))  # first minimum wins


def test_triangulation_vs_python(oracle, two_frames):
    from swarmmap_b200.matcher import FeatureVector
    f1, f2 = two_frames
    rng = np.random.default_rng(9)
    node = lambda f: (f.desc[:, 3].astype(np.int64) % 12)
    fv1, fv2 = FeatureVector(node(f1)), FeatureVector(node(f2))
    v1 = (rng.random(f1.N) < 0.8).astype(np.uint8)
    v2 = (rng.random(f2.N) < 0.8).astype(np.uint8)
    F12 = rng.normal(0, 1e-3, (3, 3)).astype(np.float32)
    F12[2, 2] = 0.05
    sf, _, s2, _ = oracle.scale_tables(1.2, 8)
    ex_, ey_ = np.float32(300.0), np.float32(150.0)
    n, out = oracle.search_for_triangulation(f1, fv1, v1, f2, fv2, v2, F12, ex_, ey_, sf, s2, False)
    F = F12.astype(np.float32)
    exp = np.full(f1.N, -1, np.int32)
    n2nodes = {int(k): fv2.feats[fv2.offsets[i]:fv2.offsets[i + 1]] for i, k in enumerate(fv2.node_ids)}
    for i, k in enumerate(fv1.node_ids):
        if int(k) not in n2nodes:
            continue
        for idx1 in fv1.feats[fv1.offsets[i]:fv1.offsets[i + 1]]:
            if not v1[idx1]:
                continue
            x1, y1 = np.float32(f1.x[idx1]), np.float32(f1.y[idx1])
            a = np.float32(np.float32(np.float32(x1 * F[0, 0]) + np.float32(y1 * F[1, 0])) + F[2, 0])
            b = np.float32(np.float32(np.float32(x1 * F[0, 1]) + np.float32(y1 * F[1, 1])) + F[2, 1])
            c = np.float32(np.float32(np.float32(x1 * F[0, 2]) + np.float32(y1 * F[1, 2])) + F[2, 2])
            best_d, best_j = TH_LOW, -1
            for idx2 in n2nodes[int(k)]:
                if not v2[idx2]:
                    continue
                d = hamming(f1.desc[idx1], f2.desc[idx2])
                if d > TH_LOW or d > best_d:
                    continue
                x2, y2, o2 = np.float32(f2.x[idx2]), np.float32(f2.y[idx2]), f2.octave[idx2]
                dx, dy = np.float32(ex_ - x2), np.float32(ey_ - y2)
                if np.float32(np.float32(dx * dx) + np.float32(dy * dy)) < np.float32(np.float32(100) * sf[o2]):
                    continue
                num = np.float32(np.float32(np.float32(a * x2) + np.float32(b * y2)) + c)
                den = np.float32(np.float32(a * a) + np.float32(b * b))
                if den == 0:
                    continue
                dsqr = np.float32(np.float32(num * num) / den)
                if float(dsqr) < 3.84 * float(s2[o2]):
                    best_d, best_j = d, int(idx2)
            exp[idx1] = best_j
    np.testing.assert_array_equal(out, exp)
    assert n == int((exp >= 0).sum()) and n > 3


def three_maxima(hist):
    """ORBmatcher::ComputeThreeMaxima, ORBmatcher.cc:1475-1506."""
    max1 = max2 = max3 = 0
    ind1 = ind2 = ind3 = -1
    for i, h in enumerate(hist):
        s = len(h)
        if s > max1:
            max3, max2, max1 = max2, max1, s
            ind3, ind2, ind1 = ind2, ind1, i
        elif s > max2:
            max3, max2 = max2, s
            ind3, ind2 = ind2, i
        elif s > max3:
            max3, ind3 = s, i
    if max2 < np.float32(0.1) * np.float32(max1):
        ind2 = ind3 = -1
    elif max3 < np.float32(0.1) * np.float32(max1):
        ind3 = -1
    return ind1, ind2, ind3


def rot_bin(a1, a2):
    rot = np.float32(a1) - np.float32(a2)
    if rot < 0:
        rot = np.float32(rot + np.float32(360.0))
    x = float(np.float32(rot * (np.float32(1.0) / np.float32(30))))
    b = int(math.copysign(math.floor(abs(x) + 0.5), x))  # C round(): halves away from zero
    return 0 if b == 30 else b


def features_in_area_levels(f, grid, x, y, r, lo, hi):
    out = get_features_in_area(f, grid, x, y, r)
    if lo > 0 or hi >= 0:  # bCheckLevels, Frame.cc:398
        out = [j for j in out if not (f.octave[j] < lo) and not (hi >= 0 and f.octave[j] > hi)]
    return out


def _params(natural, kind):
    return natural + [pytest.param(c, id=c.name) for c in matcher_cases.cases(kind)]


@pytest.mark.parametrize("inp", _params([True, False], "init"))
def test_search_for_initialization_vs_python(oracle, two_frames, inp):
    """A literal Python SearchForInitialization (ORBmatcher.cc:375-479) incl. the steal rule, the rotation histogram
    and the vbPrevMatched update: on two natural frames (inp = check_ori) and on every hand-built Init case."""
    if isinstance(inp, bool):
        f1, f2 = two_frames
        nnratio, window, check_ori = np.float32(0.9), 60, inp
        prev0 = np.stack([f1.x, f1.y], 1).astype(np.float32)
    else:
        f1, f2, window, check_ori, prev0 = inp.f1, inp.f2, inp.window, inp.check_ori, inp.prev
        nnratio = np.float32(inp.nnratio)
    n, m12, prev = oracle.search_for_initialization(f1, f2, prev0, window, float(nnratio), check_ori)
    if not isinstance(inp, bool):
        inp.reach(oracle, (n, m12, prev))
    grid = oracle.grid_csr(f2)
    INT_MAX = 2 ** 31 - 1
    match12 = np.full(f1.N, -1, np.int64)
    match21 = np.full(f2.N, -1, np.int64)
    mdist = np.full(f2.N, INT_MAX, np.int64)
    hist = [[] for _ in range(30)]
    nm = 0
    for i1 in range(f1.N):
        if f1.octave[i1] > 0:
            continue
        cand = features_in_area_levels(f2, grid, prev0[i1, 0], prev0[i1, 1], window, 0, 0)
        if not cand:
            continue
        best, best2, bi = INT_MAX, INT_MAX, -1
        for i2 in cand:
            d = hamming(f1.desc[i1], f2.desc[i2])
            if mdist[i2] <= d:
                continue
            if d < best:
                best2, best, bi = best, d, i2
            elif d < best2:
                best2 = d
        if best <= TH_LOW and np.float32(best) < np.float32(best2) * nnratio:
            if match21[bi] >= 0:
                match12[match21[bi]] = -1
                nm -= 1
            match12[i1], match21[bi], mdist[bi] = bi, i1, best
            nm += 1
            if check_ori:
                hist[rot_bin(f1.angle[i1], f2.angle[bi])].append(i1)
    if check_ori:
        keep = three_maxima(hist)
        for i in range(30):
            if i in keep:
                continue
            for idx1 in hist[i]:
                if match12[idx1] >= 0:
                    match12[idx1] = -1
                    nm -= 1
    exp_prev = prev0.copy()
    for i1 in range(f1.N):
        if match12[i1] >= 0:
            exp_prev[i1] = (f2.x[match12[i1]], f2.y[match12[i1]])
    assert n == nm and (n > 20 or not isinstance(inp, bool))
    np.testing.assert_array_equal(m12, match12)
    np.testing.assert_array_equal(prev, exp_prev)


@pytest.mark.parametrize("inp", _params([0, 1], "bow"))
def test_search_by_bow_vs_python(oracle, two_frames, inp):
    """Literal Python SearchByBoW: KeyFrame->Frame (ORBmatcher.cc:150-262) and KeyFrame<->KeyFrame (:481-597), on two
    natural frames (inp = mode) and on every hand-built BoW case."""
    from swarmmap_b200.matcher import FeatureVector
    if isinstance(inp, int):
        mode = inp
        f1, f2 = two_frames
        rng = np.random.default_rng(4)
        node = lambda f: (f.desc[:, 7].astype(np.int64) % 9)
        fv1, fv2 = FeatureVector(node(f1)), FeatureVector(node(f2))
        v1 = (rng.random(f1.N) < 0.8).astype(np.uint8)
        v2 = (rng.random(f2.N) < 0.8).astype(np.uint8)
        nnratio, check_ori = np.float32(0.75), True
    else:
        f1, f2, fv1, fv2, v1, mode = inp.f1, inp.f2, inp.fv1, inp.fv2, inp.valid1, inp.mode
        v2 = inp.valid2 if mode == 1 else np.ones(f2.N, np.uint8)
        nnratio, check_ori = np.float32(inp.nnratio), inp.check_ori
    n, out = oracle.search_by_bow(f1, fv1, v1, f2, fv2, v2 if mode == 1 else None, mode, float(nnratio), check_ori)
    if not isinstance(inp, int):
        inp.reach(oracle, (n, out, None))
    exp = np.full(f2.N if mode == 0 else f1.N, -1, np.int64)
    taken = np.zeros(f2.N, bool)
    hist = [[] for _ in range(30)]
    nm = 0
    n2nodes = {int(k): fv2.feats[fv2.offsets[i]:fv2.offsets[i + 1]] for i, k in enumerate(fv2.node_ids)}
    for i, k in enumerate(fv1.node_ids):
        if int(k) not in n2nodes:
            continue
        for idx1 in fv1.feats[fv1.offsets[i]:fv1.offsets[i + 1]]:
            if not v1[idx1]:
                continue
            b1, b2, bi = 256, 256, -1
            for idx2 in n2nodes[int(k)]:
                if taken[idx2] or (mode == 1 and not v2[idx2]):
                    continue
                d = hamming(f1.desc[idx1], f2.desc[idx2])
                if d < b1:
                    b2, b1, bi = b1, d, int(idx2)
                elif d < b2:
                    b2 = d
            ok = (b1 <= TH_LOW) if mode == 0 else (b1 < TH_LOW)
            if ok and np.float32(b1) < nnratio * np.float32(b2):
                taken[bi] = True
                if mode == 0:
                    exp[bi] = idx1
                    hist[rot_bin(f1.angle[idx1], f2.angle[bi])].append(bi)
                else:
                    exp[idx1] = bi
                    hist[rot_bin(f1.angle[idx1], f2.angle[bi])].append(int(idx1))
                nm += 1
    if check_ori:
        keep = three_maxima(hist)
        for i in range(30):
            if i in keep:
                continue
            for idx in hist[i]:
                exp[idx] = -1
                nm -= 1
    assert n == nm and (n > 10 or not isinstance(inp, int))
    np.testing.assert_array_equal(out, exp)


@pytest.mark.parametrize("inp", _params([1, 0], "window"))
def test_window_matcher_vs_python(oracle, two_frames, inp):
    """The generic windowed matcher behind the four SearchByProjection overloads, against literal Python loops:
    ratio_mode 1 = SearchByProjection(F, vpMapPoints, th) (ORBmatcher.cc:44-121: same-level ratio test, no rotation
    check, a point only blocks a slot when Observations() > 0), ratio_mode 0 = SearchByProjection(cur, last, th,
    mono) (:1223-1354: threshold only, rotation histogram over the assigned slots).  On two natural frames
    (inp = ratio_mode) and on every hand-built window case."""
    if isinstance(inp, int):
        ratio_mode = inp
        src, tgt = two_frames
        rng = np.random.default_rng(8)
        sf = oracle.scale_tables(1.2, 8)[0]
        m = src.N
        desc, angle = src.desc, src.angle
        u = (src.x + rng.normal(0, 2, m)).astype(np.float32)
        v = (src.y + rng.normal(0, 2, m)).astype(np.float32)
        valid = (rng.random(m) < 0.9).astype(np.uint8)
        blocks = (rng.random(m) < 0.7).astype(np.uint8)  # pMP->Observations() > 0
        tgt_blocked = (rng.random(tgt.N) < 0.1).astype(np.uint8)
        nnratio = np.float32(0.8)
        if ratio_mode == 1:
            lo, hi = src.octave - 1, src.octave.copy()
            radius = (np.float32(4.0) * np.float32(3.0) * sf[src.octave]).astype(np.float32)
            th_dist, check_ori = 100, False
        else:
            lo, hi = src.octave - 1, src.octave + 1
            radius = (np.float32(15.0) * sf[src.octave]).astype(np.float32)
            th_dist, check_ori = 100, True
    else:
        c = inp
        tgt, desc, angle, u, v, radius, lo, hi = c.tgt, c.desc, c.angle, c.u, c.v, c.radius, c.lo, c.hi
        valid, blocks, tgt_blocked, m = c.valid, c.blocks, c.tgt_blocked, len(c.u)
        th_dist, ratio_mode, nnratio, check_ori = c.th_dist, c.ratio_mode, np.float32(c.nnratio), c.check_ori
    n, asg = oracle.match_window(tgt, desc, u, v, radius, lo, hi, valid, blocks, th_dist, ratio_mode, float(nnratio),
                                 check_ori, angle, tgt_blocked)
    if not isinstance(inp, int):
        inp.reach(oracle, (n, asg, None))
    grid = oracle.grid_csr(tgt)
    blocked = tgt_blocked.astype(bool).copy()
    exp = np.full(tgt.N, -1, np.int64)
    hist = [[] for _ in range(30)]
    nm = 0
    for i in range(m):
        if not valid[i]:
            continue
        cand = features_in_area_levels(tgt, grid, u[i], v[i], radius[i], lo[i], hi[i])
        if not cand:
            continue
        b1, b2, l1, l2, bi = 256, 256, -1, -1, -1
        for j in cand:
            if blocked[j]:
                continue
            d = hamming(desc[i], tgt.desc[j])
            if d < b1:
                b2, l2 = b1, l1
                b1, l1, bi = d, tgt.octave[j], j
            elif d < b2:
                b2, l2 = d, tgt.octave[j]
        if b1 <= th_dist:
            if ratio_mode == 1 and l1 == l2 and np.float32(b1) > nnratio * np.float32(b2):
                continue
            exp[bi] = i
            if blocks[i]:
                blocked[bi] = True
            nm += 1
            if check_ori:
                hist[rot_bin(angle[i], tgt.angle[bi])].append(bi)
    if check_ori:
        keep = three_maxima(hist)
        for b in range(30):
            if b in keep:
                continue
            for j in hist[b]:
                exp[j] = -1
                nm -= 1
    assert n == nm and (n > 30 or not isinstance(inp, int))
    np.testing.assert_array_equal(asg, exp)
