"""A second reading of Frame::ComputeStereoMatches (ORB-SLAM2 Frame.cc:516-690) in numpy, written from the reference's
rules (the header comment of swarmmap_b200/csrc/stereo.cuh, DESIGN section 9 item 3) and not from the oracle's code.

For each left keypoint:
  1. candidates: right keypoints whose row band [floor(y - r), ceil(y + r)], r = 2 * scale(octave), holds the left
     keypoint's row (int)vL, whose octave is within +-1 of the left one and whose x lies in [uL - maxD, uL + 3],
     maxD = mbf / mb.  The best is the smallest Hamming distance, the lowest right index among equals; it must be
     below TH_HIGH = 100.
  2. an 11 x 11 SAD, each window minus its centre pixel, at the right keypoint's scaled column + incR, incR = -5..5,
     in mvImagePyramid[left octave] (blurred inside the level, the un-blurred border outside); the right column must
     satisfy scaleduR0 >= 0 and scaleduR0 + 11 < level width.  The first minimum wins and must not be at incR = +-5.
  3. a parabola through the three SADs around the minimum gives deltaR (|deltaR| > 1 is refused), then
     bestuR = scale * (scaleduR0 + incR + deltaR) and disparity = uL - bestuR, kept if 0 <= disparity < maxD;
     disparity 0 becomes 0.01 with bestuR = uL - 0.01 evaluated in double.  depth = mbf / disparity.
  4. median filter: median = the SAD at position m / 2 of the m matches sorted ascending; a match whose SAD is not
     below (1.5f * 1.4f) * median is cleared.

Every float expression is evaluated in float32, one operation at a time, in the reference's order.  C's round is half
away from zero.  Inputs are those of oracle_lib.stereo_matches; planes are the per-level bordered (19 px) composite
planes: the un-blurred buffer with the blurred level pasted inside.

The |deltaR| > 1 rule cannot fire: the minimum is the first strict one, so with a = dist1 - dist2 > 0 and
c = dist3 - dist2 >= 0 (exact integers in float32) deltaR = (a - c) / (2 (a + c)) lies in [-1/2, 1/2].  The trace keeps
the largest |deltaR| seen so that tests can check the bound.
"""
import numpy as np

F32 = np.float32
TH_HIGH = 100
BORDER = 19

OUTCOMES = ("no_candidate", "th_high", "window", "sad_edge", "delta", "disparity", "clamped", "kept", "filtered")
(NO_CANDIDATE, TH, WINDOW, SAD_EDGE, DELTA, DISPARITY, CLAMPED, KEPT, FILTERED) = range(len(OUTCOMES))

_POPCOUNT = np.array([bin(i).count("1") for i in range(256)], np.int32)


def c_round(x):
    """C's roundf (half away from zero) of float32 values; exact in float64."""
    x = np.asarray(x, F32).astype(np.float64)
    return np.copysign(np.floor(np.abs(x) + 0.5), x).astype(F32)


def hamming(a, b):
    return _POPCOUNT[np.bitwise_xor(a, b)].sum(-1)


def tally(trace, into=None):
    """Counts of each outcome and of the two flags of one trace, added into `into` (a dict) if given."""
    out = into if into is not None else {k: 0 for k in OUTCOMES + ("tie", "border")}
    counts = np.bincount(trace["outcome"], minlength=len(OUTCOMES))
    for k, c in zip(OUTCOMES, counts):
        out[k] += int(c)
    out["tie"] += int(trace["tie"].sum())
    out["border"] += int(trace["border"].sum())
    return out


def stereo_matches(kl, dl, kr, dr, planes_l, planes_r, sf, inv_sf, mbf, mb):
    """-> (u, z, kept, trace).  u / z: mvuRight / mvDepth (float32, -1 = no match); kept = matches left after the
    median filter; trace: dict of per-left-keypoint arrays:
      outcome  index into OUTCOMES (the rule that decided the keypoint)
      tie      the descriptor winner's distance was shared by another candidate
      border   the right SAD strip read outside the level (from the un-blurred border)
      dist, idx_r, scaled_ur0, bestk, sad, best_ur, disparity   intermediate values (-1 / nan where not reached)
      n_sad_min  how many of the 11 SADs equal the minimum (0 where no SAD was computed)
    and the scalars max_abs_delta, median."""
    sf, inv_sf = np.asarray(sf, F32), np.asarray(inv_sf, F32)
    mbf, mb = F32(mbf), F32(mb)
    nl, nr = len(kl), len(kr)
    uL, vL, levL = np.asarray(kl["x"], F32), np.asarray(kl["y"], F32), np.asarray(kl["octave"], np.int64)
    uR, vR, levR = np.asarray(kr["x"], F32), np.asarray(kr["y"], F32), np.asarray(kr["octave"], np.int64)
    dl, dr = np.asarray(dl, np.uint8).reshape(nl, 32), np.asarray(dr, np.uint8).reshape(nr, 32)
    n_rows = planes_l[0].shape[0] - 2 * BORDER

    u = np.full(nl, -1, F32)
    z = np.full(nl, -1, F32)
    outcome = np.full(nl, NO_CANDIDATE, np.int64)
    tie = np.zeros(nl, bool)
    border = np.zeros(nl, bool)
    best_dist = np.full(nl, -1, np.int64)
    idx_r = np.full(nl, -1, np.int64)
    scaled_ur0 = np.full(nl, np.nan, F32)
    bestk = np.full(nl, -1, np.int64)
    n_sad_min = np.zeros(nl, np.int64)
    sad_best = np.full(nl, -1, np.int64)
    disparity_out = np.full(nl, np.nan, F32)
    best_ur_out = np.full(nl, np.nan, F32)
    trace = dict(outcome=outcome, tie=tie, border=border, dist=best_dist, idx_r=idx_r, scaled_ur0=scaled_ur0,
                 bestk=bestk, n_sad_min=n_sad_min, sad=sad_best, best_ur=best_ur_out, disparity=disparity_out, max_abs_delta=0.0,
                 median=None)
    if nl == 0:
        return u, z, 0, trace

    # 1. candidates and the descriptor winner
    maxD = mbf / mb
    row = np.trunc(vL).astype(np.int64)                        # (int)vL
    minU = uL - maxD
    maxU = uL - F32(-3)
    left_ok = (row >= 0) & (row < n_rows) & ~(maxU < 0)
    r = F32(2) * sf[levR]
    maxr = np.ceil(vR + r).astype(np.int64)
    minr = np.floor(vR - r).astype(np.int64)
    cand = (left_ok[:, None] & (row[:, None] >= minr[None]) & (row[:, None] <= maxr[None]) &
            (levR[None] >= levL[:, None] - 1) & (levR[None] <= levL[:, None] + 1) &
            (uR[None] >= minU[:, None]) & (uR[None] <= maxU[:, None]))
    il, jr = np.nonzero(cand)                                   # row-major: ascending right index per left keypoint
    d = hamming(dl[il], dr[jr]).astype(np.int64)
    key = np.full(nl, np.iinfo(np.int64).max, np.int64)
    np.minimum.at(key, il, d * (1 << 20) + jr)
    has = key != np.iinfo(np.int64).max
    best_dist[has] = key[has] >> 20
    idx_r[has] = key[has] & ((1 << 20) - 1)
    n_equal = np.zeros(nl, np.int64)
    np.add.at(n_equal, il, d == best_dist[il])
    outcome[has] = TH
    won = has & (best_dist < TH_HIGH)
    tie[won] = n_equal[won] > 1

    # 2. SAD refinement, per left octave
    iw = np.nonzero(won)[0]
    scaled_ul = c_round(uL[iw] * inv_sf[levL[iw]])
    scaled_vl = c_round(vL[iw] * inv_sf[levL[iw]])
    sur0 = c_round(uR[idx_r[iw]] * inv_sf[levL[iw]])
    scaled_ur0[iw] = sur0
    width = np.array([planes_r[l].shape[1] - 2 * BORDER for l in levL[iw]], np.int64)
    height = np.array([planes_r[l].shape[0] - 2 * BORDER for l in levL[iw]], np.int64)
    iniu = (sur0 + F32(5)) - F32(5)                             # scaleduR0 + L - w
    endu = ((sur0 + F32(5)) + F32(5)) + F32(1)                  # scaleduR0 + L + w + 1
    win_ok = ~((iniu < 0) | (endu >= width.astype(F32)))
    outcome[iw[~win_ok]] = WINDOW
    iw, scaled_ul, scaled_vl, sur0, width, height = (a[win_ok] for a in (iw, scaled_ul, scaled_vl, sur0, width, height))
    n = len(iw)
    sads = np.zeros((n, 11), np.int64)
    y0 = scaled_vl.astype(np.int64) - 5
    xl0 = scaled_ul.astype(np.int64) - 5
    xr0 = sur0.astype(np.int64) - 10                            # right strip: columns of incR = -5 .. +5, +-5 px
    border[iw] = (xr0 < 0) | (xr0 + 20 >= width) | (y0 < 0) | (y0 + 10 >= height)
    span = np.arange(11)
    for lev in np.unique(levL[iw]):
        sel = np.nonzero(levL[iw] == lev)[0]
        pl, pr = np.asarray(planes_l[lev], np.int64), np.asarray(planes_r[lev], np.int64)
        rows = BORDER + y0[sel, None] + span[None]                               # (s, 11)
        cl = BORDER + xl0[sel, None] + span[None]
        cr = BORDER + xr0[sel, None] + np.arange(21)[None]
        for a, lim in ((rows, pl.shape[0]), (cl, pl.shape[1]), (cr, pr.shape[1])):
            assert a.min() >= 0 and a.max() < lim, "window outside the bordered plane"
        wl = pl[rows[:, :, None], cl[:, None, :]]                                # (s, 11, 11)
        strip = pr[rows[:, :, None], cr[:, None, :]]                             # (s, 11, 21)
        wl = wl - wl[:, 5:6, 5:6]
        for k in range(11):
            wr = strip[:, :, k:k + 11]
            sads[sel, k] = np.abs(wl - (wr - wr[:, 5:6, 5:6])).sum((1, 2))
    bk = np.argmin(sads, 1)                                     # first minimum
    bestk[iw] = bk
    n_sad_min[iw] = (sads == sads.min(1, keepdims=True)).sum(1) if n else 0
    sad_best[iw] = sads[np.arange(n), bk]
    edge = (bk == 0) | (bk == 10)
    outcome[iw[edge]] = SAD_EDGE
    keep = ~edge
    iw, bk, sads, sur0 = iw[keep], bk[keep], sads[keep], sur0[keep]

    # 3. parabola, disparity, depth
    rows_ = np.arange(len(iw))
    dist1 = sads[rows_, bk - 1].astype(F32)
    dist2 = sads[rows_, bk].astype(F32)
    dist3 = sads[rows_, bk + 1].astype(F32)
    with np.errstate(divide="ignore", invalid="ignore"):
        delta = (dist1 - dist3) / (F32(2) * ((dist1 + dist3) - F32(2) * dist2))
    if len(delta):
        trace["max_abs_delta"] = float(np.nanmax(np.abs(delta)))
    bad = (delta < -1) | (delta > 1)
    outcome[iw[bad]] = DELTA
    iw, bk, sur0, delta = iw[~bad], bk[~bad], sur0[~bad], delta[~bad]
    best_ur = sf[levL[iw]] * ((sur0 + (bk - 5).astype(F32)) + delta)
    disp = uL[iw] - best_ur
    best_ur_out[iw] = best_ur
    disparity_out[iw] = disp
    inside = (disp >= 0) & (disp < maxD)
    outcome[iw[~inside]] = DISPARITY
    iw, best_ur, disp = iw[inside], best_ur[inside], disp[inside]
    clamp = disp <= 0
    disp = np.where(clamp, F32(0.01), disp).astype(F32)
    best_ur = np.where(clamp, (uL[iw].astype(np.float64) - 0.01).astype(F32), best_ur).astype(F32)
    z[iw] = mbf / disp
    u[iw] = best_ur
    outcome[iw] = np.where(clamp, CLAMPED, KEPT)

    # 4. median filter
    m = len(iw)
    if m == 0:
        return u, z, 0, trace
    s = sad_best[iw]
    median = F32(np.sort(s)[m // 2])
    trace["median"] = int(median)
    th = (F32(1.5) * F32(1.4)) * median
    cleared = iw[~(s.astype(F32) < th)]
    u[cleared] = -1
    z[cleared] = -1
    outcome[cleared] = FILTERED
    return u, z, m - len(cleared), trace
