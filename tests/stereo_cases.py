"""Hand-built inputs of Frame::ComputeStereoMatches, one frame per rule, shared by the CPU test of the second reading
(test_oracle_stereo_independent.py) and the device test (test_gpu_stereo_geometry.py), which injects them into the
extractor's resident keypoint buffers.

Each case is one stereo frame: a synthetic image pair (make_pair) plus hand-placed left and right keypoints and
descriptors.  The images are built so that the SAD stage behaves predictably:
  * a texture mirror-symmetric about every column offset + k * period, the right view shifted by D px (right(x) =
    left(x + D)): a left keypoint on a symmetry column and a right keypoint within +-4 px of x - D give equal SADs on
    both sides of the minimum, so deltaR = 0 and the disparity is exactly D (level 0);
  * sensor noise on the right view only, mirror-symmetric as well, weak in the top half and the last 24 rows and strong
    in between, so matches in the two bands have SADs several times apart;
  * or a texture of period 4 px, where the SAD has several equal minima.
`expect[call][i]` is the outcome (stereo_ref.OUTCOMES) the rules give left keypoint i under CALLS[call]; every rule is
reached on both sides of its edge.  Keypoints stay inside the limits that keep every window read of the device kernel
within the 19-px border (the device test asserts them before any launch).
"""
import zlib

import numpy as np

import stereo_ref

F32 = np.float32
W, H = 752, 480
KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                     ("octave", "<i4"), ("class_id", "<i4")])  # cv::KeyPoint's layout
# (mbf, mb) of the calls every case is run under: maxD = 16, maxD = 1 exactly, maxD = the next float above 1
CALLS = [(16.0, 1.0), (1.0, 1.0), (float(np.nextafter(F32(1), F32(2))), 1.0)]


def _tri(x, period):
    t = np.mod(x, 2 * period)
    return np.abs(t - period)


def make_pair(D=4, seed=1, noise=(1, 12), period=48, offset=0, periodic4=False):
    """(left, right) uint8 H x W images, see the module docstring."""
    rng = np.random.default_rng(seed)
    x = np.arange(W)
    if periodic4:
        tex = rng.integers(0, 256, (H, 4)).astype(np.int32)
        il, ir = x % 4, (x + D) % 4
    else:
        tex = rng.integers(0, 256, (H, period + 1)).astype(np.int32)
        il, ir = _tri(x - offset, period), _tri(x + D - offset, period)
    y = np.arange(H)
    amp = np.where((y >= H // 2) & (y < H - 24), noise[1], noise[0])[:, None]
    nz = np.round(rng.uniform(-1, 1, tex.shape) * amp).astype(np.int32)
    left = tex[:, il]
    right = np.clip(tex + nz, 0, 255)[:, ir]
    return left.astype(np.uint8), right.astype(np.uint8)


class Case:
    def __init__(self, name, sf, **pair):
        self.name, self.pair, self.sf = name, pair, np.asarray(sf, F32)
        self.rng = np.random.default_rng(zlib.crc32(name.encode()))
        self.left, self.right = [], []          # (x, y, octave, desc)
        self.expect = {0: {}, 1: {}, 2: {}}
        self.needs_planes = None                 # plane-dependent completion (see clamp_near_zero)
        for i in range(6):                       # distractors: unreachable rows, they only move the indices
            self.right.append((F32(40 + 100 * i), F32(H - 6), 0, self.desc()))

    def desc(self):
        return self.rng.integers(0, 256, 32, dtype=np.uint8)

    @staticmethod
    def flip(d, k):
        bits = np.unpackbits(d)
        bits[:k] ^= 1
        return np.packbits(bits)

    def kp(self, xs, ys, lev):
        """Level pixel (xs, ys) of octave lev in level-0 units, as the extractor writes it."""
        return F32(xs) * self.sf[lev], F32(ys) * self.sf[lev]

    def add_left(self, x, y, lev, d, expect=None, calls=(0,)):
        self.left.append((F32(x), F32(y), lev, d))
        if expect is not None:
            for c in calls:
                self.expect[c][len(self.left) - 1] = expect
        return len(self.left) - 1

    def add_right(self, x, y, lev, d, at=None):
        at = len(self.right) if at is None else at
        while len(self.right) < at:
            self.right.append((F32(40 + 7 * len(self.right)), F32(H - 6), 0, self.desc()))
        self.right.insert(at, (F32(x), F32(y), lev, d))
        return at

    def fillers(self, n=10):
        """n ordinary matches in the noisy bottom half: they raise the frame's median SAD, so that matches with the
        larger SADs of border reads survive the median filter."""
        D = self.pair.get("D", 4)
        for k in range(n):
            d = self.desc()
            x, y = 100 + 50 * k, 300 + 18 * k
            self.add_left(x, y, 0, d)
            self.add_right(x - D + 1, y, 0, self.flip(d, 5))

    def arrays(self):
        def pack(lst):
            k = np.zeros(len(lst), KP_DTYPE)
            d = np.zeros((len(lst), 32), np.uint8)
            for i, (x, y, o, dd) in enumerate(lst):
                k[i] = (x, y, 31.0, 0.0, 1.0, o, -1)
                d[i] = dd
            return k, d
        return pack(self.left) + pack(self.right)


def build_cases(sf):
    sf = np.asarray(sf, F32)
    cases = []
    K, NC, T, WIN, EDGE, DISP, CL, FIL = ("kept", "no_candidate", "th_high", "window", "sad_edge", "disparity",
                                           "clamped", "filtered")

    # descriptor tie: the lowest right index wins the packed (dist << 16 | j) minimum
    c = Case("tie", sf, D=4, seed=11)
    d = c.desc()
    i = c.add_left(300, 100, 0, d, K)                      # good match at the lower index
    c.add_right(298, 100, 0, c.flip(d, 12), at=7)
    c.add_right(289, 100, 0, c.flip(d, 12), at=8)
    c.tie_cases = [(i, 7)]
    d = c.desc()
    i = c.add_left(400, 160, 0, d, EDGE)                   # the far one at the lower index (same warp lane, j and j+32)
    c.add_right(389, 160, 0, c.flip(d, 12), at=9)
    c.add_right(398, 160, 0, c.flip(d, 12), at=41)
    c.tie_cases.append((i, 9))
    d = c.desc()
    i = c.add_left(500, 220, 0, d, K)                      # no tie: distances 12 and 11
    c.add_right(489, 220, 0, c.flip(d, 12))
    j = c.add_right(498, 220, 0, c.flip(d, 11))
    c.no_tie = [(i, j)]
    cases.append(c)

    # TH_HIGH: 99 is accepted, 100 is not
    c = Case("th_high", sf, D=4, seed=12)
    d = c.desc()
    c.add_left(300, 100, 0, d, K)
    c.add_right(298, 100, 0, c.flip(d, 99))
    d = c.desc()
    c.add_left(400, 200, 0, d, T)
    c.add_right(398, 200, 0, c.flip(d, 100))
    cases.append(c)

    # octave band +-1, at level 0, 3 and 7
    c = Case("octave", sf, D=4, seed=13)
    row = 30
    for lev, ro, e in ((0, 1, K), (0, 2, NC), (3, 2, K), (3, 4, K), (3, 1, NC), (3, 5, NC), (7, 6, K), (7, 5, NC)):
        xs, ys = int(round(300 / sf[lev])) + row // 30, int(round(row / sf[lev]))
        shift = int(round(4 / sf[lev]))
        d = c.desc()
        x, y = c.kp(xs, ys, lev)
        c.add_left(x, y, lev, d, e)
        c.add_right(c.kp(xs - shift, ys, lev)[0], y, ro, c.flip(d, 5))
        row += 50
    cases.append(c)

    # row band [floor(y - r), ceil(y + r)] with r = 2 * 1.2 (right octave 1)
    c = Case("rows", sf, D=4, seed=14)
    c.row_edges = []
    for k, (dy, e) in enumerate(((2.7, K), (3.5, NC), (-2.7, K), (-3.5, NC))):
        row = 60 + 50 * k
        d = c.desc()
        i = c.add_left(300 + 20 * k, row, 0, d, e)
        c.add_right(298 + 20 * k, F32(row) + F32(dy), 1, c.flip(d, 5))
        c.row_edges.append((i, row, dy))
    cases.append(c)

    # uR in [uL - maxD, uL + 3] (maxD = 16)
    c = Case("u_range", sf, D=1, seed=15)
    for k, (mk, e) in enumerate(((lambda u: u + F32(3), K),
                                 (lambda u: np.nextafter(u + F32(3), F32(1e9)), NC),
                                 (lambda u: u - F32(16), EDGE),
                                 (lambda u: np.nextafter(u - F32(16), F32(-1e9)), NC))):
        row = 60 + 50 * k
        d = c.desc()
        uL = F32(300 + 20 * k)
        c.add_left(uL, row, 0, d, e)
        c.add_right(mk(uL), row, 0, c.flip(d, 5))
    cases.append(c)

    # window check scaleduR0 >= 0 and scaleduR0 + 11 < w; scaleduR0 <= 9 reads the un-blurred border
    c = Case("window", sf, D=4, seed=16)
    d = c.desc()
    x, y = c.kp(3, 40, 1)
    c.add_left(x, y, 1, d, WIN)                            # scaleduR0 = round(-0.65 / 1.2) = -1
    c.add_right(F32(-0.65), y, 2, c.flip(d, 5))
    row = 100
    for s in (0, 1, 9, 10):
        for r in range(3):
            d = c.desc()
            c.add_left(4 + s, row, 0, d, K if s >= 9 else None)
            c.add_right(s, row, 0, c.flip(d, 5))
            row += 12
    for s, e in ((W - 12, K), (W - 11, WIN)):
        d = c.desc()
        c.add_left(s + 4, row, 0, d, e)
        c.add_right(s, row, 0, c.flip(d, 5))
        row += 12
    for yy in (0, 1, H - 2, H - 1):                       # rows outside the level
        d = c.desc()
        c.add_left(200 + yy % 100, yy, 0, d, K)
        c.add_right(196 + yy % 100, yy, 0, c.flip(d, 5))
    c.fillers()
    cases.append(c)

    # disparity 0 on symmetry columns: the clamp (bestuR = uL - 0.01 in double)
    c = Case("clamp", sf, D=0, seed=17, offset=24)
    for k in range(1, 7):
        d = c.desc()
        x = 24 + 48 * k + (48 if k > 3 else 0)
        c.add_left(x, 240 + 30 * k, 0, d)                   # noisy band: a median above the near-zero SADs
        c.add_right(x + (k % 3) - 1, 240 + 30 * k, 0, c.flip(d, 5))
    c.needs_planes = clamp_near_zero
    cases.append(c)

    # disparity exactly 1 = maxD under CALLS[1]: refused there, kept under CALLS[0] and CALLS[2]
    c = Case("max_disparity", sf, D=1, seed=18)
    for k in range(1, 4):
        d = c.desc()
        c.add_left(48 * (k + 2), 40 + 40 * k, 0, d)
        for call, e in ((0, K), (1, DISP), (2, K)):
            c.expect[call][len(c.left) - 1] = e
        c.add_right(48 * (k + 2) - 1, 40 + 40 * k, 0, c.flip(d, 5))
    cases.append(c)

    # one match: the median is its own SAD
    c = Case("one_match", sf, D=4, seed=19)
    d = c.desc()
    c.add_left(300, 100, 0, d, K)
    c.add_right(298, 100, 0, c.flip(d, 3))
    cases.append(c)

    # duplicated left keypoints: SADs [a, a, b, b] with b > 2.1 a; the median is element m / 2 = b, so all are kept
    c = Case("median_ties", sf, D=4, seed=20)
    for y in (100, 100, 400, 400):
        d = np.full(32, y % 256, np.uint8)
        c.add_left(300, y, 0, d, K)
    c.add_right(298, 100, 0, np.full(32, 100, np.uint8))
    c.add_right(298, 400, 0, np.full(32, 400 % 256, np.uint8))
    cases.append(c)

    # noise-free views: every SAD is 0, the median is 0 and the filter clears everything
    c = Case("median_zero", sf, D=4, seed=21, noise=(0, 0))
    for k in range(4):
        d = c.desc()
        c.add_left(200 + 60 * k, 60 + 60 * k, 0, d, FIL)
        c.add_right(198 + 60 * k, 60 + 60 * k, 0, c.flip(d, 5))
    cases.append(c)

    # period-4 texture: equal SAD minima, the first one wins
    c = Case("sad_ties", sf, D=0, seed=22, periodic4=True, noise=(2, 2))
    for k in range(8):
        d = c.desc()
        c.add_left(200 + 40 * k, 40 + 25 * k, 0, d)
        c.add_right(200 + 40 * k - 2 - (k % 2), 40 + 25 * k, 0, c.flip(d, 5))
    cases.append(c)
    return cases


def _differs(v):
    v = F32(v)
    return F32(np.float64(v) - 0.01) != v - F32(0.01)


def clamp_near_zero(case, planes_l, planes_r, sf, inv_sf):
    """Adds left keypoints at x < 0.125 whose bestuR equals their own x, so the clamp's uL - 0.01 in double and in
    float differ.  First pass: keypoints at x = 0.05 on every fourth row; the SAD stage depends on x only through
    round(x) = 0, so a second keypoint at x = bestuR of the first gets the same bestuR and disparity 0."""
    probe = Case("probe", sf)
    probe.right = []
    rows = list(range(8, H - 8, 4))
    for y in rows:
        d = probe.desc()
        probe.add_left(0.05, y, 0, d)
        probe.add_right(1.0, y, 0, d)
    kl, dl, kr, dr = probe.arrays()
    u, _, _, tr = stereo_ref.stereo_matches(kl, dl, kr, dr, planes_l, planes_r, sf, inv_sf, *CALLS[0])
    bestur = tr["best_ur"]
    picked = [k for k in range(len(rows)) if 0.01 < bestur[k] < 0.125 and _differs(bestur[k])]
    picked = sorted(picked, key=lambda k: tr["sad"][k])[:3]   # the smallest SADs pass the frame's median filter
    for k in picked:
        y = rows[k]
        case.add_left(bestur[k], y, 0, dl[k], "clamped")
        case.add_right(1.0, y, 0, dr[k])
    case.near_zero = len(picked)
