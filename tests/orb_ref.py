"""Float64 reference of the extractor's last stage, checked keypoint by keypoint: level coordinates, size, response,
orientation (IC_Angle, reference Fast_gpu.cu:403-460) and rBRIEF (calcOrb_kernel, Orb_gpu.cu:67-100).

TEST INFRASTRUCTURE, numpy only.  It reads the planes the keypoints were described from: per level the bordered
(19 px) un-blurred plane, the blurred ROI and, when the extractor kept one, the FAST score map.  The GPU gives them
through ORBextractor.debug_plane(frame, level, 0 / 1 / 2), the CPU oracle through Extractor.level(level, 0 / 1 / 2).

Bounds (derived from the float32 arithmetic both implementations use, not measured):
- angle: CUDA documents atan2f at 3 ulp (7.2e-7 rad at pi); the float32 roundings of + 2 pi and of x 180 / pi add
  2.4e-7 and 2.7e-7 rad; CV_PI_F differs from pi by 8.7e-8, which the + 2 pi and the x 180 / CV_PI_F scale by up to 4.
  Together about 1.5e-6 rad; ANGLE_TOL_RAD allows 4e-6.
- descriptor: the rotation of a pattern point uses float32 radians (2.4e-7 rad), cosf / sinf at 2 ulp and float32
  products and sums: under 2e-5 px at the pattern's largest radius of 18.4 px.  A bit may therefore differ from the
  float64 rotation only where one of its two points lies within HALF_PX_TOL = 1e-4 px of a rounding boundary
  (a half-integer).  Any other differing bit is a wrong descriptor.
"""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EDGE = 19          # border of the un-blurred planes (EDGE_THRESHOLD, ORBextractor.cc:78)
HALF_PATCH = 15    # ORBextractor.cc:77
PATCH = 31
ANGLE_TOL_RAD = 4e-6
HALF_PX_TOL = 1e-4


def load_pattern():
    txt = open(os.path.join(ROOT, "oracle", "orb_pattern_data.inc")).read()
    body = txt[txt.index("{") + 1:txt.index("};")]
    vals = np.array([int(v) for v in re.findall(r"-?\d+", body)], np.int64)
    assert len(vals) == 1024
    return vals.reshape(512, 2)  # (x, y) per sample point; bit i compares point 2i with point 2i + 1


def make_umax():
    """Disc half-widths of the orientation patch (ORBextractor.cc:380-404)."""
    umax = np.zeros(HALF_PATCH + 1, np.int64)
    vmax = int(np.floor(np.float32(HALF_PATCH * np.sqrt(np.float32(2)) / 2 + 1)))
    vmin = int(np.ceil(np.float32(HALF_PATCH * np.sqrt(np.float32(2)) / 2)))
    for v in range(vmax + 1):
        umax[v] = int(np.rint(np.sqrt(float(HALF_PATCH * HALF_PATCH - v * v))))
    v0 = 0
    for v in range(HALF_PATCH, vmin - 1, -1):
        while umax[v0] == umax[v0 + 1]:
            v0 += 1
        umax[v] = v0
        v0 += 1
    return umax


PATTERN = load_pattern()
UMAX = make_umax()


def _disc(umax):
    vv, uu = np.mgrid[-HALF_PATCH:HALF_PATCH + 1, -HALF_PATCH:HALF_PATCH + 1]
    inside = np.abs(uu) <= np.asarray(umax, np.int64)[np.abs(vv)]
    return vv[inside], uu[inside]


def ref_angles(plain, lx, ly, umax=UMAX):
    """Float64 orientation in degrees, [0, 360), of level-coordinate points (lx, ly) on a bordered un-blurred plane:
    exact int64 intensity moments over the radius-15 disc, then atan2(m01, m10)."""
    dv, du = _disc(umax)
    win = plain[(ly[:, None] + EDGE + dv[None, :]), (lx[:, None] + EDGE + du[None, :])].astype(np.int64)
    m10 = win @ du
    m01 = win @ dv
    return np.mod(np.degrees(np.arctan2(m01.astype(np.float64), m10.astype(np.float64))), 360.0)


def ref_descriptors(blur, lx, ly, angle_deg, pattern=PATTERN):
    """rBRIEF bits of points (lx, ly) on a blurred ROI with the pattern rotated in float64 by angle_deg (each point's
    own angle).  -> (bits (n, 256) uint8, ambiguous (n, 256) bool).  A bit is ambiguous when a rotated coordinate
    of one of its points is within HALF_PX_TOL of a half-integer, where float32 rounding may pick either pixel.
    Asserts that every pixel the rounding could pick lies inside the ROI."""
    rad = np.deg2rad(np.asarray(angle_deg, np.float64))
    a, b = np.cos(rad)[:, None], np.sin(rad)[:, None]
    px, py = pattern[:, 0].astype(np.float64)[None, :], pattern[:, 1].astype(np.float64)[None, :]
    fx = px * a - py * b
    fy = px * b + py * a
    amb_pt = (np.abs(np.abs(fx - np.floor(fx)) - 0.5) <= HALF_PX_TOL) | \
             (np.abs(np.abs(fy - np.floor(fy)) - 0.5) <= HALF_PX_TOL)
    X = lx[:, None] + np.rint(fx).astype(np.int64)   # round half to even (__float2int_rn, lrintf)
    Y = ly[:, None] + np.rint(fy).astype(np.int64)
    h, w = blur.shape
    xlo, xhi = lx[:, None] + np.floor(fx), lx[:, None] + np.ceil(fx)
    ylo, yhi = ly[:, None] + np.floor(fy), ly[:, None] + np.ceil(fy)
    bad = (xlo < 0) | (xhi >= w) | (ylo < 0) | (yhi >= h)
    if bad.any():
        k = int(np.nonzero(bad.any(1))[0][0])
        raise AssertionError(f"rBRIEF sample outside the {w}x{h} blurred ROI for the keypoint at level ({lx[k]}, {ly[k]})")
    vals = blur[Y, X].astype(np.int16)
    bits = (vals[:, 0::2] < vals[:, 1::2]).astype(np.uint8)
    return bits, amb_pt[:, 0::2] | amb_pt[:, 1::2]


def check_keypoints(kps, desc, planes, blurs, sf, scores=None, umax=UMAX, pattern=PATTERN, what="frame"):
    """Checks every keypoint of one frame against the float64 reference and raises AssertionError naming the first
    keypoint that fails.  kps: KP_DTYPE array, desc: (n, 32) uint8; planes[l]: bordered un-blurred plane,
    blurs[l]: blurred ROI, scores[l]: FAST score map (or None); sf: scale factor per level.
    -> dict(n, max_angle_err_rad, ambiguous_bits)."""
    kps = np.asarray(kps)
    desc = np.asarray(desc, np.uint8).reshape(-1, 32)
    assert len(kps) == len(desc), what
    sf = np.asarray(sf, np.float32)
    stats = {"n": len(kps), "max_angle_err_rad": 0.0, "ambiguous_bits": 0}
    if len(kps) == 0:
        return stats
    assert (kps["class_id"] == -1).all(), f"{what}: class_id != -1"
    oct_ = kps["octave"]
    assert oct_.min() >= 0 and oct_.max() < len(planes), f"{what}: octave out of range"
    for o in np.unique(oct_):
        idx = np.nonzero(oct_ == o)[0]
        k = kps[idx]
        s = sf[o]
        lx = np.rint(k["x"].astype(np.float64) / np.float64(s)).astype(np.int64)
        ly = np.rint(k["y"].astype(np.float64) / np.float64(s)).astype(np.int64)
        for name, lv, v in (("x", lx, k["x"]), ("y", ly, k["y"])):
            back = lv.astype(np.float32) if o == 0 else lv.astype(np.float32) * s
            bad = np.nonzero(back.view(np.uint32) != v.view(np.uint32))[0]
            assert len(bad) == 0, f"{what}: keypoint {idx[bad[0]]} (octave {o}) {name}={v[bad[0]]!r} is not a level pixel x {s!r}"
        size = np.float32(int(np.float32(PATCH) * s))
        bad = np.nonzero(k["size"] != size)[0]
        assert len(bad) == 0, f"{what}: keypoint {idx[bad[0]]} (octave {o}) size {k['size'][bad[0]]} != {size}"
        if scores is not None:
            resp = scores[o][ly, lx].astype(np.float32)
            bad = np.nonzero(k["response"] != resp)[0]
            assert len(bad) == 0, f"{what}: keypoint {idx[bad[0]]} (octave {o}) response {k['response'][bad[0]]} != score map {resp[bad[0]]}"
        # orientation against float64
        ref = ref_angles(planes[o], lx, ly, umax)
        d = np.abs(np.deg2rad(k["angle"].astype(np.float64)) - np.deg2rad(ref))
        d = np.minimum(d, 2 * np.pi - d)
        j = int(np.argmax(d))
        stats["max_angle_err_rad"] = max(stats["max_angle_err_rad"], float(d[j]))
        assert d[j] <= ANGLE_TOL_RAD, \
            f"{what}: keypoint {idx[j]} (octave {o}, level ({lx[j]}, {ly[j]})) angle {k['angle'][j]!r} deg vs float64 {ref[j]!r}: {d[j]:.3e} rad"
        # descriptor from the keypoint's own angle
        bits, amb = ref_descriptors(blurs[o], lx, ly, k["angle"].astype(np.float64), pattern)
        got = np.unpackbits(desc[idx], axis=1, bitorder="little")
        wrong = (got != bits) & ~amb
        if wrong.any():
            r, c = np.argwhere(wrong)[0]
            raise AssertionError(f"{what}: keypoint {idx[r]} (octave {o}, level ({lx[r]}, {ly[r]}), angle {k['angle'][r]!r}) "
                                 f"descriptor byte {c // 8} bit {c % 8} differs from float64 rBRIEF "
                                 f"({int(wrong.sum())} unexplained bits on {int(wrong.any(1).sum())} keypoints)")
        stats["ambiguous_bits"] += int(amb.sum())
    return stats


def check_extractor_frame(ex, frame, kps, desc, score=True, what=None):
    """check_keypoints on the planes a GPU ORBextractor kept for `frame` of its last call (score maps only when the
    handle was made with debug_score=True)."""
    nl = ex.GetLevels()
    planes = [ex.debug_plane(frame, l, 0) for l in range(nl)]
    blurs = [ex.debug_plane(frame, l, 1) for l in range(nl)]
    scores = [ex.debug_plane(frame, l, 2) for l in range(nl)] if score else None
    return check_keypoints(kps, desc, planes, blurs, ex.GetScaleFactors(), scores, what=what or f"frame {frame}")


def merge(total, stats):
    """Accumulates check_keypoints results: counts add up, the angle error is the maximum."""
    for k, v in stats.items():
        total[k] = max(total.get(k, 0.0), v) if k.startswith("max_") else total.get(k, 0) + v
    return total
