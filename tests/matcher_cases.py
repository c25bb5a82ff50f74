"""Inputs for the monocular matchers whose greedy loop runs through one resolve (swarmmap_b200/csrc/match.cu
resolve_body): SearchForInitialization, the windowed SearchByProjection forms and both SearchByBoW forms.

`random_frame` is the tie-heavy synthetic frame generator.  `hand_built()` returns small deterministic frame pairs,
each built so that one rule of the resolve sits on its edge: candidate rows of 31..65 and > 1000 entries with
equal-distance ties whose enumeration order differs from index order, speculative batches whose first conflict falls
at a chosen position, conflicts on the second best only, Init steals, the float32 ratio tests, the TH_LOW / TH_HIGH
thresholds, rotation bins at their rounding half-points and ComputeThreeMaxima at its 10 % cut.  Descriptors get
exact Hamming distances by flipping chosen bits of a source descriptor.  Each case carries `reach(oracle, result)`,
a host-side assertion on the oracle's answer that the case really reaches its edge."""
import numpy as np

from swarmmap_b200.matcher import FeatureVector, Frame

W, H = 640, 400
TH_LOW, TH_HIGH = 50, 100
INT_MAX = 2 ** 31 - 1
RATIOS = (0.6, 0.7, 0.75, 0.8, 0.9, 1.5)  # every nnratio the ORB-SLAM2 call sites use, and one above 1
BOUNDS = (0.0, 0.0, 640.0, 480.0)  # 64 x 48 grid cells of exactly 10 x 10 px


def random_frame(rng, n, bits=None, bounds=(0.0, 0.0, float(W), float(H)), cluster=False, base=None):
    """Synthetic frame: tie-heavy when `bits` is small (descriptors differ in few bits), clustered positions.  Frames
    meant to match each other share `base` (1 x 32 uint8), the descriptor their bits are flipped from."""
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
        if base is None:
            base = rng.integers(0, 256, (1, 32), dtype=np.uint8)
        flip = np.zeros((n, 256), np.uint8)
        for i in range(n):
            flip[i, rng.integers(0, 256, bits)] = 1
        desc = base ^ np.packbits(flip, axis=1)
    return Frame(xy[:, 0], xy[:, 1], octave, angle, desc, bounds)


# ------------------------------------------------------------------------------------------------ descriptors

def hamming(a, b):
    return int(np.unpackbits(np.asarray(a, np.uint8) ^ np.asarray(b, np.uint8)).sum())


def flip(d, bits):
    b = np.unpackbits(np.asarray(d, np.uint8).copy())
    b[list(bits)] ^= 1
    return np.packbits(b)


def at(rng, s, d, avoid=()):
    """A descriptor at Hamming distance exactly d from s, differing from it in none of the bits `avoid`."""
    pool = np.setdiff1d(np.arange(256), np.asarray(list(avoid), np.int64))
    return flip(s, rng.choice(pool, d, replace=False))


def two_way(rng, sa, da, sb, db):
    """A descriptor at distance da from sa and db from sb."""
    D = np.nonzero(np.unpackbits(sa ^ sb))[0]
    k2 = da + len(D) - db
    assert k2 % 2 == 0 and 0 <= k2 // 2 <= min(len(D), da), (da, db, len(D))
    inside = rng.choice(D, k2 // 2, replace=False)
    outside = rng.choice(np.setdiff1d(np.arange(256), D), da - k2 // 2, replace=False)
    t = flip(sa, np.concatenate([inside, outside]))
    assert hamming(t, sa) == da and hamming(t, sb) == db
    return t


def f32(x):
    return np.float32(x)


def ratio_disagreements(ratio, rule, th):
    """(best, second) pairs, best <= th <= 256 and best <= second, where the reference's float32 ratio comparison and
    the exact one disagree.  rule "lt": accept when float(best) < fl(ratio_f * second) (Init, SearchByBoW); rule "gt":
    reject when float(best) > fl(ratio_f * second) (the same-level test of SearchByProjection(F, points))."""
    from fractions import Fraction
    r = f32(ratio)
    out = []
    for b in range(th + 1):
        for s in range(b, 257):
            p = f32(r * f32(s))
            exact = Fraction(float(r)) * s
            if rule == "lt" and (f32(b) < p) != (b < exact):
                out.append((b, s))
            if rule == "gt" and (f32(b) > p) != (b > exact):
                out.append((b, s))
    return out


def half_point_rots():
    """Angle differences rot (a1 - a2 >= 0) for which fl(rot * fl(1/30)) is exactly k + 0.5: C round() sends them up,
    round-half-to-even would send even k down.  At most one per k = 0..11 (k = 2 and 9 have none)."""
    f = f32(1.0) / f32(30)
    out = {}
    for k in range(12):
        centre = f32(30 * (k + 0.5))
        x = centre
        for _ in range(64):  # walk down in ulps, then up
            if f32(x * f) == f32(k + 0.5):
                out[k] = x
                break
            x = np.nextafter(x, f32(0))
        if k not in out:
            x = centre
            for _ in range(64):
                x = np.nextafter(x, f32(1000))
                if f32(x * f) == f32(k + 0.5):
                    out[k] = x
                    break
    return out


def rot_bin_c(rot):
    """Bin of an angle difference under C round (half away from zero) -- used only to state what a case reaches."""
    rot = f32(rot)
    if rot < 0:
        rot = f32(rot + f32(360.0))
    x = float(f32(rot * (f32(1.0) / f32(30))))
    b = int(np.floor(x + 0.5))
    return 0 if b == 30 else b


# ------------------------------------------------------------------------------------------------ cases

class Case:
    """kind "init": f1, f2, prev, window, nnratio, check_ori.  kind "window": tgt and the match_window arguments
    (desc, u, v, radius, lo, hi, valid, blocks, angle, tgt_blocked, th_dist, ratio_mode, nnratio, check_ori).  kind
    "bow": f1, fv1, valid1, f2, fv2, valid2 (None for KeyFrame->Frame), mode, nnratio, check_ori."""

    def __init__(self, name, kind, reach=None, **kw):
        self.name, self.kind, self._reach = name, kind, reach
        self.__dict__.update(kw)

    def __repr__(self):
        return self.name

    def run_oracle(self, oracle):
        """-> (nmatches, match array, vbPrevMatched or None)."""
        if self.kind == "init":
            n, m12, prev = oracle.search_for_initialization(self.f1, self.f2, self.prev.copy(), self.window, self.nnratio,
                                                            self.check_ori)
            return n, m12, prev
        if self.kind == "window":
            n, asg = oracle.match_window(self.tgt, self.desc, self.u, self.v, self.radius, self.lo, self.hi, self.valid,
                                         self.blocks, self.th_dist, self.ratio_mode, self.nnratio, self.check_ori,
                                         self.angle, self.tgt_blocked)
            return n, asg, None
        n, out = oracle.search_by_bow(self.f1, self.fv1, self.valid1, self.f2, self.fv2, self.valid2, self.mode,
                                      self.nnratio, self.check_ori)
        return n, out, None

    def reach(self, oracle, result):
        if self._reach is not None:
            self._reach(self, oracle, result)


def _frame(x, y, octave, angle, desc, bounds=BOUNDS):
    n = len(x)
    return Frame(np.asarray(x, np.float32), np.asarray(y, np.float32), np.asarray(octave, np.int32).reshape(n),
                 np.asarray(angle, np.float32).reshape(n), np.asarray(desc, np.uint8).reshape(n, 32), bounds)


def _cell(cx, cy, k=0):
    """A point inside grid cell (cx, cy) of BOUNDS; k staggers several points of one cell along x."""
    return 10.0 * cx + 0.5 + 0.25 * k, 10.0 * cy + 0.5


class Scene:
    """Targets placed on the 10 px grid and source rows with explicit windows; realised as a window, Init or BoW case."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.t = []   # (x, y, octave, angle, desc, blocked, node)
        self.r = []   # dict(desc, u, v, r, lo, hi, valid, blocks, angle, node)

    def src(self):
        return self.rng.integers(0, 256, 32, dtype=np.uint8)

    def tgt(self, x, y, desc, octave=0, angle=0.0, blocked=0, node=0):
        self.t.append((x, y, octave, angle, desc, blocked, node))
        return len(self.t) - 1

    def row(self, desc, u, v, r, lo=-1, hi=-1, valid=1, blocks=1, angle=0.0, node=0):
        self.r.append(dict(desc=desc, u=u, v=v, r=r, lo=lo, hi=hi, valid=valid, blocks=blocks, angle=angle, node=node))
        return len(self.r) - 1

    def _targets(self):
        t = self.t
        return _frame([a[0] for a in t], [a[1] for a in t], [a[2] for a in t], [a[3] for a in t],
                      np.array([a[4] for a in t], np.uint8).reshape(len(t), 32))

    def window(self, name, th_dist=TH_HIGH, ratio_mode=0, nnratio=0.8, check_ori=False, reach=None):
        R = self.r
        col = lambda k, dt: np.array([r[k] for r in R], dt)
        return Case(name, "window", reach, tgt=self._targets(), desc=np.array([r["desc"] for r in R], np.uint8).reshape(-1, 32),
                    u=col("u", np.float32), v=col("v", np.float32), radius=col("r", np.float32), lo=col("lo", np.int32),
                    hi=col("hi", np.int32), valid=col("valid", np.uint8), blocks=col("blocks", np.uint8),
                    angle=col("angle", np.float32), tgt_blocked=np.array([a[5] for a in self.t], np.uint8),
                    th_dist=th_dist, ratio_mode=ratio_mode, nnratio=nnratio, check_ori=check_ori)

    def init(self, name, window, nnratio=0.9, check_ori=False, reach=None):
        """Rows become F1's keypoints (octave 0 when valid, 1 when not), windows centred on vbPrevMatched."""
        R = self.r
        assert all(r["r"] == window for r in R) and all(a[2] == 0 for a in self.t)
        f1 = _frame([r["u"] for r in R], [r["v"] for r in R], [0 if r["valid"] else 1 for r in R],
                    [r["angle"] for r in R], np.array([r["desc"] for r in R], np.uint8).reshape(-1, 32))
        prev = np.stack([f1.x, f1.y], 1).astype(np.float32).reshape(-1, 2)
        return Case(name, "init", reach, f1=f1, f2=self._targets(), prev=np.ascontiguousarray(prev), window=window,
                    nnratio=nnratio, check_ori=check_ori)

    def bow(self, name, mode, nnratio=0.75, check_ori=False, reach=None):
        """Rows become the KeyFrame's features, targets F's; each feature sits in the vocabulary node given to it."""
        R = self.r
        f1 = _frame([1.0] * len(R), [1.0] * len(R), [0] * len(R), [r["angle"] for r in R],
                    np.array([r["desc"] for r in R], np.uint8).reshape(-1, 32))
        f2 = self._targets()
        fv1 = FeatureVector(np.array([r["node"] for r in R], np.int64))
        fv2 = FeatureVector(np.array([a[6] for a in self.t], np.int64))
        valid1 = np.array([r["valid"] for r in R], np.uint8)
        valid2 = (1 - np.array([a[5] for a in self.t], np.uint8)) if mode == 1 else None
        return Case(name, "bow", reach, f1=f1, fv1=fv1, valid1=valid1, f2=f2, fv2=fv2, valid2=valid2, mode=mode,
                    nnratio=nnratio, check_ori=check_ori)


def grid_candidates(oracle, tgt, u, v, r, lo=-1, hi=-1):
    """Frame::GetFeaturesInArea through the oracle's grid: the candidates of one window, in enumeration order."""
    import ctypes as C
    fr, keep = oracle.make_frame(tgt.x, tgt.y, tgt.octave, tgt.angle, tgt.desc, tgt.bounds)
    L = oracle.lib()
    g = L.orc_grid_build(C.byref(fr))
    out = np.zeros(max(tgt.N, 1), np.int32)
    try:
        L.orc_grid_query.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int,
                                     C.c_void_p, C.c_int]
        n = L.orc_grid_query(g, C.byref(fr), float(u), float(v), float(r), int(lo), int(hi),
                             out.ctypes.data_as(C.c_void_p), tgt.N)
    finally:
        L.orc_grid_destroy(g)
    return out[:n]


# ---- independent rows: each row has private candidates at the given distances, in enumeration order

def _region(i):
    """Cell of the i-th private region: every other cell, so windows of radius < 10 px never reach a neighbour."""
    return 2 * (i % 32), 2 * (i // 32)


def independent(seed, specs):
    """specs: per row dict(d=[distances], lv=[levels] (default 0), rot=angle difference of the first candidate,
    valid=1, blocks=1).  The row's window (radius 4 px, levels unfiltered) holds exactly its candidates, in list
    order; in BoW form each row owns one node.  Returns the Scene and per row the target indices."""
    sc = Scene(seed)
    tids = []
    for i, sp in enumerate(specs):
        cx, cy = _region(i)
        s = sc.src()
        rot = f32(sp.get("rot", 0.0))
        # a1 - a2 == rot exactly; -0.0 comes from -0.0 - 0.0
        a1, a2 = (rot, f32(0.0)) if rot >= 0 else (f32(0.0), f32(-rot))
        ids = []
        for k, d in enumerate(sp["d"]):
            x, y = _cell(cx, cy, k)
            desc = (~s).astype(np.uint8) if d == 256 else at(sc.rng, s, d)
            ids.append(sc.tgt(x, y, desc, octave=sp.get("lv", [0] * len(sp["d"]))[k], angle=a2 if k == 0 else 0.0,
                              blocked=sp.get("tb", [0] * len(sp["d"]))[k], node=i))
        u, v = _cell(cx, cy, 0)
        sc.row(s, u + 1.0, v, 4.0, valid=sp.get("valid", 1), blocks=sp.get("blocks", 1), angle=a1, node=i)
        tids.append(ids)
    return sc, tids


def _expect_rows(case, result, rows_tids, accepted):
    """Reach helper: row i took its first candidate exactly where accepted[i]."""
    n, out, _ = result
    for i, (ids, acc) in enumerate(zip(rows_tids, accepted)):
        if case.kind == "window" or (case.kind == "bow" and case.mode == 0):
            got = out[ids[0]] == i
        else:
            got = out[i] == ids[0]
        assert bool(got) == bool(acc), (case.name, i, acc)


def threshold_cases():
    cases = []
    far = [180]
    specs = [dict(d=[50] + far), dict(d=[51] + far), dict(d=[49] + far)]
    for mode, acc in ((0, [1, 0, 1]), (1, [0, 0, 1])):  # SearchByBoW: `<= TH_LOW` KeyFrame->Frame, `< TH_LOW` KF<->KF
        sc, tids = independent(100 + mode, specs)
        cases.append(sc.bow(f"th_low_bow{mode}", mode, 0.75,
                            reach=lambda c, o, r, t=tids, a=acc: _expect_rows(c, r, t, a)))
    sc, tids = independent(102, specs)
    cases.append(sc.init("th_low_init", 4, 0.9, reach=lambda c, o, r, t=tids: _expect_rows(c, r, t, [1, 0, 1])))
    specs = [dict(d=[100, 250]), dict(d=[101, 250]), dict(d=[99, 250])]
    for rm in (0, 1):
        sc, tids = independent(103 + rm, specs)
        cases.append(sc.window(f"th_high_window_rm{rm}", TH_HIGH, rm, 0.8,
                               reach=lambda c, o, r, t=tids: _expect_rows(c, r, t, [1, 0, 1])))
    return cases


def ratio_cases():
    """Every (best, second) pair where float32 and exact arithmetic disagree, one private row each."""
    cases = []
    for ratio in RATIOS:
        lt = [p for p in ratio_disagreements(ratio, "lt", TH_LOW)]
        gt = [p for p in ratio_disagreements(ratio, "gt", TH_HIGH)]
        # 0.75 is exact in binary: no pair disagrees, and no row is built for it
        tag = str(ratio).replace(".", "")

        def rows(pairs):
            return [dict(d=[b, s]) for b, s in pairs]

        def acc_lt(pairs, strict_th):
            return [(b < TH_LOW if strict_th else b <= TH_LOW) and f32(b) < f32(f32(ratio) * f32(s)) for b, s in pairs]

        if lt:
            # the float32 rule rejects every one of these pairs: the exact one would accept them
            assert not any(acc_lt(lt, False)) and all(b < float(f32(ratio)) * s for b, s in lt)
            sc, tids = independent(200 + int(ratio * 100), rows(lt))
            cases.append(sc.init(f"ratio_{tag}_init", 4, ratio,
                                 reach=lambda c, o, r, t=tids: _expect_rows(c, r, t, [0] * len(t))))
            for mode in (0, 1):
                sc, tids = independent(300 + int(ratio * 100) + mode, rows(lt))
                cases.append(sc.bow(f"ratio_{tag}_bow{mode}", mode, ratio,
                                    reach=lambda c, o, r, t=tids: _expect_rows(c, r, t, [0] * len(t))))
        if gt:
            # equal levels: the same-level test applies; float32 accepts, the exact comparison would reject
            sc, tids = independent(400 + int(ratio * 100), rows(gt))
            cases.append(sc.window(f"ratio_{tag}_window_rm1", TH_HIGH, 1, ratio,
                                   reach=lambda c, o, r, t=tids: _expect_rows(c, r, t, [1] * len(t))))
    return cases


def second_best_cases():
    """best == second, P and Q at the second-best distance on different levels, a second best at distance 256."""
    cases = []
    specs = [dict(d=[20, 20], lv=[0, 0]), dict(d=[20, 256]), dict(d=[30, 31, 256], lv=[0, 1, 0]),
             dict(d=[24, 20, 24], lv=[0, 0, 1]),   # P (before the winner) is the second best: same level -> rejected
             dict(d=[24, 20, 24], lv=[1, 0, 0]),   # P on another level: the ratio test does not apply -> accepted
             dict(d=[20], lv=[0])]                 # no second best at all (256 / INT_MAX)
    sc, tids = independent(500, specs)
    # levels: the winner's is 0, and SearchByProjection(F, points) tests the ratio only on equal levels
    for s in sc.r:
        s["lo"], s["hi"] = -1, 1

    def reach_rm1(c, o, r, t=tids):
        n, asg, _ = r
        assert asg[t[0][0]] == -1 and asg[t[1][0]] == 1 and asg[t[2][0]] == 2  # tie: 20 > 0.8 * 20, same level
        assert asg[t[3][1]] == -1 and asg[t[4][1]] == 4 and asg[t[5][0]] == 5

    cases.append(sc.window("second_best_window_rm1", TH_HIGH, 1, 0.8, reach=reach_rm1))
    for mode in (0, 1):
        sc2, t2 = independent(501 + mode, specs)
        cases.append(sc2.bow(f"second_best_bow{mode}", mode, 0.75,
                             reach=lambda c, o, r, t=t2: _expect_rows(c, r, t, [0, 1, 0, 0, 0, 1])))
    sc3, t3 = independent(503, [dict(d=sp["d"]) for sp in specs])  # Init: every candidate on level 0
    cases.append(sc3.init("second_best_init", 4, 0.9,
                          reach=lambda c, o, r, t=t3: _expect_rows(c, r, t, [0, 1, 0, 0, 0, 1])))
    return cases


# ---- long candidate rows

def _block_row(sc, cx0, cy0, n, tie, pq, levels01):
    """One row whose window holds exactly n targets in a 4 x 4-cell block (up to 6 per cell).  Targets are inserted in
    shuffled order, so index order and enumeration order (column-major cells, ascending index inside a cell) differ.
    tie: the two targets at the minimum distance are enumerated in the opposite order of their indices, the first
    one enumerated has the higher index.  pq: winner in the middle, P before it and Q after it at the second-best
    distance, P on the winner's level, Q on the other.  Returns (row, winner index, enumeration order)."""
    slots = [(cx0 + (j // 6) // 4, cy0 + (j // 6) % 4, j % 6) for j in range(n)]
    order = sc.rng.permutation(n)
    s = sc.src()
    base = len(sc.t)
    # index of slot order[k] = base + k
    idx_of_slot = np.empty(n, np.int64)
    idx_of_slot[order] = base + np.arange(n)
    enum = sorted(range(n), key=lambda j: (slots[j][0], slots[j][1], idx_of_slot[j]))  # slot ids in enumeration order
    dist = {j: int(sc.rng.integers(40, 90)) for j in range(n)}
    lv = {j: int(sc.rng.integers(0, 2)) if levels01 else 0 for j in range(n)}
    win = None
    if tie:
        pairs = [(a, b) for a in range(n) for b in range(a + 1, n) if idx_of_slot[enum[a]] > idx_of_slot[enum[b]]]
        a, b = max(pairs, key=lambda p: (p[1] - p[0], p[1]))  # far apart in the row: the later one past lane 31
        dist[enum[a]] = dist[enum[b]] = 20
        lv[enum[a]], lv[enum[b]] = 0, 1 if levels01 else 0
        win = enum[a]
    if pq:
        w, p, q = n // 2, 1, n - 2
        dist[enum[w]], dist[enum[p]], dist[enum[q]] = 20, 24, 24
        lv[enum[w]], lv[enum[p]], lv[enum[q]] = 0, 0, 1 if levels01 else 0
        win = enum[w]
    for k in range(n):
        j = order[k]
        x, y = _cell(*slots[j][:2], slots[j][2])
        sc.tgt(x, y, at(sc.rng, s, dist[j]), octave=lv[j])
    u, v = 10.0 * cx0 + 17.0, 10.0 * cy0 + 17.0
    row = sc.row(s, u, v, 18.0, lo=-1, hi=1 if levels01 else -1)
    return row, int(idx_of_slot[win]), [int(idx_of_slot[j]) for j in enum]


COUNTS = (31, 32, 33, 64, 65)


def long_row_cases():
    cases = []
    for kind in ("window_rm0", "window_rm1", "init"):
        sc = Scene(600 + len(cases))
        info = []
        for i, n in enumerate(COUNTS):
            for pq in (False, True):
                if kind == "init" and pq:
                    continue
                k = 2 * i + pq
                row, win, enum = _block_row(sc, 6 * (k % 10), 6 * (k // 10), n, not pq, pq, kind != "init")
                info.append((row, n, win, enum, pq))

        def reach(c, o, r, info=info):
            n_, out, _ = r
            for row, n, win, enum, pq in info:
                if c.kind == "init":
                    got = grid_candidates(o, c.f2, c.f1.x[row], c.f1.y[row], c.window, 0, 0)
                    assert out[row] == win  # ratio 1.5: the tie passes, the first enumerated wins
                else:
                    got = grid_candidates(o, c.tgt, c.u[row], c.v[row], c.radius[row], c.lo[row], c.hi[row])
                    if c.ratio_mode == 1 and pq:
                        assert out[win] == -1  # P, on the winner's level, is the second best
                    else:
                        assert out[win] == row  # the first of the tied targets in enumeration order wins
                assert len(got) == n and list(got) == enum and list(got) != sorted(got)
        if kind == "init":
            for r in sc.r:
                r["r"] = 18.0
            cases.append(sc.init("long_rows_init", 18, 1.5, reach=reach))  # ratio 1.5: ties at the minimum pass
        else:
            cases.append(sc.window(f"long_rows_{kind}", TH_HIGH, int(kind[-1]), 0.8, reach=reach))
    # the same ties in KF->Frame BoW nodes (enumeration = ascending index there)
    specs = []
    for n in COUNTS:
        d = [int(x) for x in np.random.default_rng(n).integers(40, 90, n)]
        d[3] = d[n - 1] = 20
        specs.append(dict(d=d))
    sc, tids = independent(650, specs)
    cases.append(sc.bow("long_rows_bow0", 0, 1.5, reach=lambda c, o, r, t=tids: _expect_rows(c, r, [x[3:] for x in t],
                                                                                                [1] * len(t))))
    return cases


def whole_frame_cases():
    """One window covering the whole target (> 1000 candidates), ties enumerated against index order; plus a
    4000-keypoint KITTI-sized target."""
    cases = []
    for n, bounds, name in ((1200, BOUNDS, "whole_frame_1200"), (4000, (0.0, 0.0, 1241.0, 376.0), "kitti_4000")):
        rng = np.random.default_rng(n)
        s = rng.integers(0, 256, 32, dtype=np.uint8)
        xmax, ymax = bounds[2] * 63.4 / 64, bounds[3] * 47.4 / 48  # inside the last grid cell
        x = rng.uniform(bounds[0], xmax, n).astype(np.float32)
        y = rng.uniform(bounds[1], ymax, n).astype(np.float32)
        dist = rng.integers(30, 120, n)
        # the tie: a high index in the first column, a low index in the last
        hi_i, lo_i = n - 1, 0
        x[hi_i], x[lo_i] = bounds[0] + 0.5, xmax
        dist[hi_i] = dist[lo_i] = 10
        desc = np.array([at(rng, s, int(d)) for d in dist], np.uint8)
        octave = np.zeros(n, np.int32)
        octave[lo_i] = 1  # the same-level ratio test does not apply to the tie
        tgt = Frame(x, y, octave, np.zeros(n, np.float32), desc, bounds)
        m = 3
        others = [rng.integers(0, 256, 32, dtype=np.uint8) for _ in range(m - 1)]
        rows = np.array([s] + others, np.uint8)
        u = np.full(m, (bounds[2] - bounds[0]) / 2, np.float32)
        v = np.full(m, (bounds[3] - bounds[1]) / 2, np.float32)
        radius = np.array([2000.0, 2000.0, 30.0], np.float32)

        def reach(c, o, r, hi_i=hi_i, lo_i=lo_i, n=n):
            got = grid_candidates(o, c.tgt, c.u[0], c.v[0], c.radius[0])
            assert len(got) == n and list(got).index(hi_i) < list(got).index(lo_i)
            assert r[1][hi_i] == 0 and r[1][lo_i] != 0

        for rm in (0, 1):
            cases.append(Case(f"{name}_rm{rm}", "window", reach, tgt=tgt, desc=rows, u=u, v=v, radius=radius,
                              lo=np.full(m, -1, np.int32), hi=np.full(m, -1, np.int32), valid=np.ones(m, np.uint8),
                              blocks=np.ones(m, np.uint8), angle=np.zeros(m, np.float32),
                              tgt_blocked=np.zeros(n, np.uint8), th_dist=TH_HIGH, ratio_mode=rm, nnratio=0.9,
                              check_ori=rm == 0))
    return cases


# ---- speculative batches

def chain_cases():
    """Row k's best target is taken by row k - 1, for 40 rows: every speculative batch commits one row."""
    cases = []
    L = 41
    # window: row k sees c_k (distance 2) and c_{k+1} (distance 4); c_0 is blocked before the call
    sc = Scene(700)
    s = [sc.src()]
    for k in range(L):
        s.append(flip(s[-1], [128 + 2 * k, 129 + 2 * k]))
    c = []
    for k in range(L + 1):
        x = 14.0 * k + 6.0
        c.append(sc.tgt(x, 100.5, flip(s[k], [2, 5]), blocked=int(k == 0)))
    for k in range(L):
        sc.row(s[k], 14.0 * k + 12.0, 100.5, 9.0)

    def reach_window(cs, o, r):
        asg = r[1]
        for k in range(L):
            got = grid_candidates(o, cs.tgt, cs.u[k], cs.v[k], cs.radius[k])
            assert list(got) == [c[k], c[k + 1]]
            assert hamming(cs.desc[k], cs.tgt.desc[c[k]]) < hamming(cs.desc[k], cs.tgt.desc[c[k + 1]])
            assert asg[c[k + 1]] == k  # its best (c_k) went to row k - 1
    cases.append(sc.window("chain40_window", TH_HIGH, 0, 0.8, reach=reach_window))

    # BoW: one node; row k and c_j sit on a path of the descriptor space, distance 2 + 2 |j - k| (ratio 0.75 passes)
    sc = Scene(701)
    s = [sc.src()]
    for k in range(L + 1):
        s.append(flip(s[-1], [128 + 2 * k, 129 + 2 * k]))
    for k in range(L):
        sc.row(s[k], 0.0, 0.0, 1.0, node=7)
    cb = [sc.tgt(1.0, 1.0, flip(s[j], [3, 9]), node=7) for j in range(1, L + 1)]  # c_1 .. c_L (no c_0)

    def reach_bow(cs, o, r):
        out = r[1]
        for k in range(L):
            if cs.mode == 0:
                assert out[cb[k]] == k
            else:
                assert out[k] == cb[k]
    for mode in (0, 1):
        cases.append(sc.bow(f"chain40_bow{mode}", mode, 0.75, reach=reach_bow))
    return cases


def conflict_position_cases():
    """40 independent rows, except that the row at list position p finds its best taken by row p - 1 (p = 1, 30, 31:
    inside the first batch; p = 32: the first row of the next batch).  Window, BoW and Init forms."""
    cases = []
    for p in (1, 30, 31, 32):
        specs = [dict(d=[12, 60]) for _ in range(40)]
        for kind in ("window", "bow", "init"):
            sc, tids = independent(800 + p, specs)
            # row p sees row p - 1's target T at distance 13 (T at 12 from row p - 1) and its own at 30
            T = tids[p - 1][0]
            sp = sc.r[p - 1]["desc"]
            s = at(sc.rng, sp, 1, avoid=np.nonzero(np.unpackbits(sp ^ sc.t[T][4]))[0])
            sc.r[p]["desc"] = s
            own = tids[p][0]
            x, y = sc.t[own][0], sc.t[own][1]
            sc.t[own] = (x, y, 0, 0.0, at(sc.rng, s, 30), 0, p)
            sc.t[tids[p][1]] = (sc.t[tids[p][1]][0], y, 0, 0.0, at(sc.rng, s, 90), 0, p)
            # put T into row p's window / node: move row p onto row p - 1's region, its targets next to T
            sc.r[p].update(u=sc.r[p - 1]["u"], v=sc.r[p - 1]["v"], node=p - 1)
            tx, ty = sc.t[T][0], sc.t[T][1]
            for k, j in enumerate(tids[p]):
                sc.t[j] = (tx + 0.5 + 0.25 * k, ty) + sc.t[j][2:6] + (p - 1,)

            def reach(c, o, r, p=p, T=T, own=own):
                out = r[1]
                if c.kind in ("init", "bow"):  # Init steals only at a smaller distance: 13 > 12
                    assert out[p - 1] == T and out[p] == own
                else:
                    assert out[T] == p - 1 and out[own] == p
            if kind == "window":
                cases.append(sc.window(f"conflict_at_{p}_window", TH_HIGH, 0, 0.8, reach=reach))
            elif kind == "bow":
                cases.append(sc.bow(f"conflict_at_{p}_bow1", 1, 0.75, reach=reach))
            else:
                cases.append(sc.init(f"conflict_at_{p}_init", 4, 0.9, reach=reach))
    return cases


def second_only_cases():
    """Row p - 1 takes row p's SECOND best S; row p's best B is untouched.  With S present row p fails its ratio
    test (20 vs 22); once S is gone its second best is 40 and it passes."""
    cases = []
    for kind in ("window_rm1", "bow0", "bow1", "init"):
        sc = Scene(900 + len(cases))
        info = []
        for i, p in enumerate((1, 17, 31, 34, 40)):
            while len(sc.r) < p - 1:  # filler rows with private targets
                cx, cy = _region(len(sc.r) + 40 * i)
                s = sc.src()
                x, y = _cell(cx, cy)
                sc.tgt(x, y, at(sc.rng, s, 15), node=1000 + len(sc.r))
                sc.row(s, x + 1.0, y, 4.0, node=1000 + len(sc.r))
            sp = sc.src()
            s = at(sc.rng, sp, 12)
            D = np.nonzero(np.unpackbits(sp ^ s))[0]
            cx, cy = _region(200 + i)
            x, y = _cell(cx, cy)
            node = 500 + i
            B = sc.tgt(x, y, at(sc.rng, s, 20, avoid=D), node=node)
            S = sc.tgt(x + 0.25, y, two_way(sc.rng, s, 22, sp, 10), node=node)
            F = sc.tgt(x + 0.5, y, at(sc.rng, s, 40, avoid=D), node=node)
            sc.row(sp, x + 1.0, y, 4.0, node=node)
            sc.row(s, x + 1.0, y, 4.0, node=node)
            info.append((p - 1, p, B, S, F))
            assert hamming(sp, sc.t[B][4]) == 32 and hamming(sp, sc.t[F][4]) == 52

        def reach(c, o, r, info=info):
            out = r[1]
            for q, p, B, S, F in info:
                if c.kind == "window" or (c.kind == "bow" and c.mode == 0):
                    assert out[S] == q and out[B] == p
                else:
                    assert out[q] == S and out[p] == B
        if kind == "window_rm1":
            cases.append(sc.window("second_only_window_rm1", TH_HIGH, 1, 0.8, reach=reach))
        elif kind.startswith("bow"):
            cases.append(sc.bow(f"second_only_{kind}", int(kind[-1]), 0.75, reach=reach))
        else:
            cases.append(sc.init("second_only_init", 4, 0.9, reach=reach))
    return cases


def list_cases():
    """Lists of 31, 32, 33 and 64 valid non-empty rows, interleaved with invalid rows and rows whose window is empty;
    the last valid row finds its best taken by the valid row before it."""
    cases = []
    for nvalid in (31, 32, 33, 64):
        specs = []
        kinds = []
        for i in range(nvalid):
            specs.append(dict(d=[15, 70]))
            kinds.append("v")
            if i % 3 == 1:
                specs.append(dict(d=[10], valid=0))
                kinds.append("invalid")
            if i % 4 == 2:
                specs.append(dict(d=[]))
                kinds.append("empty")
        sc, tids = independent(1000 + nvalid, specs)
        vrows = [i for i, k in enumerate(kinds) if k == "v"]
        a, b = vrows[-2], vrows[-1]
        T = tids[a][0]
        sb = at(sc.rng, sc.r[a]["desc"], 1, avoid=np.nonzero(np.unpackbits(sc.r[a]["desc"] ^ sc.t[T][4]))[0])
        sc.r[b].update(desc=sb, u=sc.r[a]["u"], v=sc.r[a]["v"], node=a)
        for k, j in enumerate(tids[b]):
            sc.t[j] = (sc.t[T][0] + 0.5 + 0.25 * k, sc.t[T][1], 0, 0.0, at(sc.rng, sb, 30 + 40 * k), 0, a)

        def reach(c, o, r, kinds=kinds, tids=tids, a=a, b=b, T=T):
            out = r[1]
            if c.kind == "window":
                for i, k in enumerate(kinds):
                    if k == "empty":
                        assert len(grid_candidates(o, c.tgt, c.u[i], c.v[i], c.radius[i])) == 0
                    if k == "invalid":
                        assert len(grid_candidates(o, c.tgt, c.u[i], c.v[i], c.radius[i])) == 1 and out[tids[i][0]] == -1
                assert out[T] == a and out[tids[b][0]] == b
            else:
                assert out[a] == T and out[b] == tids[b][0]
        assert kinds.count("v") == nvalid
        cases.append(sc.window(f"list_{nvalid}_window", TH_HIGH, 0, 0.8, reach=reach))
        cases.append(sc.bow(f"list_{nvalid}_bow1", 1, 0.75, reach=reach))
    return cases


# ---- Init steals

def steal_cases():
    """One target stolen at distances d, d - 1, d - 2 (rows 0, 1, 2: one batch; rows 0, 40, 80: three batches); an
    equal-distance later row that must not steal; a stolen source whose rotation bin is pruned."""
    cases = []
    for spread, name in ((1, "steal_chain_batch"), (40, "steal_chain_across")):
        for ori in (False, True):
            n = 2 * spread + 2 if spread > 1 else 4
            specs = [dict(d=[25], rot=60.0) for _ in range(max(n, 90))]
            sc, tids = independent(1100 + spread + ori, specs)
            r0, r1, r2 = 0, spread, 2 * spread
            eq = r2 + 1
            s0 = sc.r[r0]["desc"]
            T = tids[r0][0]
            X = np.nonzero(np.unpackbits(s0 ^ sc.t[T][4]))[0]
            assert len(X) == 25
            s1 = flip(s0, [X[0]])
            s2 = flip(s1, [X[1]])
            for r, s in ((r1, s1), (r2, s2), (eq, s2.copy())):
                sc.r[r].update(desc=s, u=sc.r[r0]["u"], v=sc.r[r0]["v"])
                for j in tids[r]:  # the row's own target leaves the window: only T is left
                    sc.t[j] = (sc.t[j][0], sc.t[j][1] + 5.0) + sc.t[j][2:]
            if ori:
                # row 0's match falls in bin 8, alone: pruned after row 1 stole its target (it must not count down)
                sc.r[r0]["angle"] = f32(240.0)
                sc.t[T] = sc.t[T][:3] + (f32(0.0),) + sc.t[T][4:]

            def reach(c, o, r, r0=r0, r1=r1, r2=r2, eq=eq, T=T):
                n_, m12, prev = r
                assert m12[r0] == -1 and m12[r1] == -1 and m12[r2] == T and m12[eq] == -1
                d = [hamming(c.f1.desc[k], c.f2.desc[T]) for k in (r0, r1, r2, eq)]
                assert d == [25, 24, 23, 23]
                assert np.array_equal(prev[r0], c.prev[r0]) and np.array_equal(prev[r2], [c.f2.x[T], c.f2.y[T]])
            cases.append(sc.init(f"{name}{'_ori' if ori else ''}", 4, 0.9, check_ori=ori, reach=reach))
    return cases


# ---- rotation

def _rot_case(seed, rots, name, kind="window", blocks=None, reach=None, shared=None):
    specs = [dict(d=[30], rot=float(r)) for r in rots]
    if blocks is not None:
        for sp, b in zip(specs, blocks):
            sp["blocks"] = b
    sc, tids = independent(seed, specs)
    if shared:  # rows sharing one target (non-blocking window sources): same descriptor, same window
        first = shared[0]
        for r in shared[1:]:
            sc.r[r].update(desc=sc.r[first]["desc"].copy(), u=sc.r[first]["u"], v=sc.r[first]["v"])
            for j in tids[r]:
                sc.t[j] = (sc.t[j][0], sc.t[j][1] + 5.0) + sc.t[j][2:]
    if kind == "window":
        return sc.window(name, TH_HIGH, 0, 0.8, check_ori=True, reach=reach)
    if kind == "init":
        return sc.init(name, 4, 0.9, check_ori=True, reach=reach)
    return sc.bow(name, int(kind[-1]), 0.75, check_ori=True, reach=reach)


def rotation_cases():
    cases = []
    hp = half_point_rots()
    assert {0, 4, 6, 8, 10} <= set(hp)
    # half-points of k = 0 (-> bin 1, not 0) decide which bins survive: bins 4 (10), 7 (8), 0 (6), 1 (5 half-points)
    rots = [120.0] * 10 + [210.0] * 8 + [0.0] * 6 + [hp[0]] * 5

    def reach_half(c, o, r):
        bins = [rot_bin_c(x) for x in rots]
        assert bins.count(1) == 5 and bins.count(0) == 6
        assert float(f32(f32(hp[0]) * (f32(1.0) / f32(30)))) == 0.5
        out = r[1]
        assert int((out >= 0).sum()) == 24 and r[0] == 24  # bin 1 (the half-points) is pruned
    for kind in ("window", "init", "bow0", "bow1"):
        cases.append(_rot_case(1200 + len(cases), rots, f"rot_half_points_{kind}", kind, reach=reach_half))
    # every even-k half-point, -0.0, a tiny negative difference (+360 rounds to 360.0f: bin 12), the other bins
    rots2 = [hp[k] for k in sorted(hp) if k % 2 == 0] * 3 + [-0.0] * 4 + [-1e-6] * 5 + [f32(359.99)] * 2 + [f32(345.0)] * 3

    def reach_edges(c, o, r):
        assert rot_bin_c(-1e-6) == 12 and f32(f32(-1e-6) + f32(360.0)) == f32(360.0) and rot_bin_c(-0.0) == 0
    for kind in ("window", "init", "bow0"):
        cases.append(_rot_case(1210 + len(cases), rots2, f"rot_edges_{kind}", kind, reach=reach_edges))
    # ComputeThreeMaxima: max2 / max3 exactly 0.1 * max1 (kept: the cut is `<`), and ties among the top counts
    for top in (10, 20, 30):
        rr = [90.0] * top + [180.0] * (top // 10) + [270.0] * (top // 10) + [330.0] * (top // 10 - 1 if top > 10 else 0)

        def reach_cut(c, o, r, top=top):
            assert f32(0.1) * f32(top) == f32(top // 10)
            assert r[0] == top + 2 * (top // 10)  # max2 == max3 == 0.1 * max1 are kept, the fourth bin is not
        cases.append(_rot_case(1220 + top, rr, f"three_maxima_cut_{top}", reach=reach_cut))
    cases.append(_rot_case(1250, [30.0] * 5 + [60.0] * 5 + [90.0] * 5 + [120.0] * 5 + [150.0] * 4, "three_maxima_ties",
                           reach=_matches(15)))  # four bins of 5: the first three are kept
    # two non-blocking window sources on one target, both in a pruned bin: nmatches drops by two
    rr = [90.0] * 10 + [180.0] * 8 + [270.0] * 6 + [150.0, 150.0]

    def reach_two(c, o, r):
        T = 24  # row 24's own target: rows 24 and 25 share it
        assert r[0] == 24 and r[1][T] == -1
    cases.append(_rot_case(1260, rr, "rot_two_nonblocking_pruned", "window", blocks=[1] * 24 + [0, 0], shared=[24, 25],
                           reach=reach_two))
    # the same with the two sources 1024 rows apart (one pruning thread meets both events, one after the other), and
    # 999 invalid rows with empty windows between them
    specs = ([dict(d=[30], rot=150.0, blocks=0)] + [dict(d=[30], rot=90.0)] * 10 + [dict(d=[30], rot=180.0)] * 8
             + [dict(d=[30], rot=270.0)] * 6 + [dict(d=[], valid=0)] * 999 + [dict(d=[30], rot=150.0, blocks=0)])
    sc, tids = independent(1261, specs)
    sc.r[1024].update(desc=sc.r[0]["desc"].copy(), u=sc.r[0]["u"], v=sc.r[0]["v"])
    sc.t[tids[1024][0]] = (sc.t[tids[1024][0]][0], sc.t[tids[1024][0]][1] + 5.0) + sc.t[tids[1024][0]][2:]

    def reach_far(c, o, r):
        assert len(c.u) == 1025 and r[0] == 24 and r[1][0] == -1  # 26 accepted, both events on target 0 pruned
    cases.append(sc.window("rot_two_nonblocking_pruned_1024_apart", TH_HIGH, 0, 0.8, check_ori=True, reach=reach_far))
    return cases


def overwrite_cases():
    """Non-blocking sources (Observations() == 0) taking the same target: the later one overwrites."""
    rr = [0.0] * 6

    def reach(c, o, r):
        asg = r[1]
        assert asg[0] == 2 and r[0] == 6  # rows 0, 1, 2 all matched target 0; the last write wins
    return [_rot_case(1300, rr, "nonblocking_overwrite", "window", blocks=[0, 0, 1, 1, 1, 1], shared=[0, 1, 2],
                      reach=reach)]


def _matches(n):
    def reach(c, o, r):
        assert r[0] == n, (c.name, r[0], n)
    return reach


def degenerate_cases():
    cases = []
    sc, _ = independent(1400, [dict(d=[20], valid=0) for _ in range(5)])
    cases.append(sc.window("no_valid_rows_window", reach=_matches(0)))
    cases.append(sc.init("no_valid_rows_init", 4, reach=_matches(0)))
    cases.append(sc.bow("no_valid_rows_bow0", 0, reach=_matches(0)))
    sc, _ = independent(1401, [dict(d=[]) for _ in range(40)])
    sc.tgt(600.5, 400.5, sc.src())
    cases.append(sc.window("every_window_empty", reach=_matches(0)))
    cases.append(sc.init("every_window_empty_init", 4, reach=_matches(0)))
    sc, _ = independent(1402, [dict(d=[]) for _ in range(3)])
    assert not sc.t
    cases.append(sc.window("zero_keypoint_target", reach=_matches(0)))
    cases.append(sc.bow("zero_keypoint_target_bow1", 1, reach=_matches(0)))
    sc, _ = independent(1403, [dict(d=[20, 40])])
    cases.append(sc.window("single_row", reach=_matches(1)))
    cases.append(sc.init("single_row_init", 4, reach=_matches(1)))
    cases.append(sc.bow("single_row_bow0", 0, reach=_matches(1)))
    return cases


def hand_built():
    return (long_row_cases() + whole_frame_cases() + chain_cases() + conflict_position_cases() + second_only_cases()
            + list_cases() + steal_cases() + second_best_cases() + threshold_cases() + ratio_cases() + rotation_cases()
            + overwrite_cases() + degenerate_cases())


_CASES = None


def cases(kind=None):
    global _CASES
    if _CASES is None:
        _CASES = hand_built()
    return [c for c in _CASES if kind is None or c.kind == kind]
