"""A second reading, in numpy, of Frame::isInFrustum (Frame.cc:316-375), MapPoint::PredictScale (MapPoint.cc:476-485)
and the projections of the two tracking SearchByProjection calls (ORBmatcher.cc:44-121 with Tracking.cc:964-1006, and
ORBmatcher.cc:1223-1354 with bMono = true).  Vectorised per call; every float expression is evaluated in float32 in
the reference's order, with the cv::Mat rules DESIGN.md section 2 freezes (see oracle/orb_oracle_frustum.cpp):
Pc = R P + t with float products and sums; Ow = -R^T t, cv::norm and Mat::dot in double.

`log` of a float is glibc's logf, called through ctypes: numpy's float32 log is a different implementation and may
differ from it in the last bit, which moves PredictScale's level at its thresholds.

is_in_frustum returns, per point, the rule that decided it (RULES) and the intermediate values."""
import ctypes
import ctypes.util

import numpy as np

RULES = ("behind", "u_out", "v_out", "dist_small", "dist_large", "angle", "in_view")
F32 = np.float32

_logf = ctypes.CDLL(ctypes.util.find_library("m")).logf
_logf.argtypes = [ctypes.c_float]
_logf.restype = ctypes.c_float


def logf(a):
    a = np.asarray(a, F32)
    return np.array([_logf(float(x)) for x in a.ravel()], F32).reshape(a.shape)


def gemm_small(T, P):
    """Rcw * P + tcw, cv::gemm's small-matrix path: float products and sums left to right, then + t (float)."""
    T = np.asarray(T, F32)
    P = np.asarray(P, F32).reshape(-1, 3)
    out = np.empty_like(P)
    for r in range(3):
        acc = T[r, 0] * P[:, 0]
        acc = acc + T[r, 1] * P[:, 1]
        acc = acc + T[r, 2] * P[:, 2]
        out[:, r] = acc + T[r, 3]
    return out


def camera_centre(T):
    """Ow = -Rcw.t() * tcw on the generic path: double products and sums, left to right, then float."""
    T = np.asarray(T, F32)
    Ow = np.zeros(3, F32)
    for c in range(3):
        acc = 0.0
        for k in range(3):
            acc += float(np.float64(T[k, c]) * np.float64(T[k, 3]))
        Ow[c] = F32(-1.0 * acc)
    return Ow


def predict_scale(max_distance, dist, log_sf, nlevels):
    """ratio = max / dist (float), ceil(logf(ratio) / logScaleFactor) in float, clamped to [0, nlevels - 1];
    NaN -> 0, +inf -> nlevels - 1 (the reference's int conversion is undefined there)."""
    with np.errstate(all="ignore"):
        ratio = np.asarray(max_distance, F32) / np.asarray(dist, F32)
        q = np.ceil(logf(ratio) / F32(log_sf))
    lvl = np.where(np.isnan(q), 0, np.clip(np.nan_to_num(q, nan=0.0, posinf=1e9, neginf=-1e9), 0, nlevels - 1))
    return lvl.astype(np.int32)


def is_in_frustum(T, K, bounds4, pos, normal, min_d, max_d, log_sf, nlevels, cos_limit=0.5):
    """-> dict(in_view, u, v, view_cos, level, rule, Pc, invz, u_raw, v_raw, dist, min_dist, max_dist, view_cos_raw,
    ratio).  rule[i] indexes RULES.  u, v, view_cos, level are 0 where the point is not in view."""
    T = np.asarray(T, F32)[:3, :4]
    fx, fy, cx, cy = [F32(k) for k in K]
    b = np.asarray(bounds4, F32)
    pos = np.asarray(pos, F32).reshape(-1, 3)
    normal = np.asarray(normal, F32).reshape(-1, 3)
    n = len(pos)
    with np.errstate(all="ignore"):
        Pc = gemm_small(T, pos)
        invz = F32(1.0) / Pc[:, 2]
        u = fx * Pc[:, 0] * invz + cx
        v = fy * Pc[:, 1] * invz + cy
        Ow = camera_centre(T)
        PO = pos - Ow
        s = np.zeros(n)
        for k in range(3):
            s = s + PO[:, k].astype(np.float64) * PO[:, k].astype(np.float64)
        dist = np.sqrt(s).astype(F32)
        mind = F32(0.8) * np.asarray(min_d, F32)
        maxd = F32(1.2) * np.asarray(max_d, F32)
        dot = np.zeros(n)
        for k in range(3):
            dot = dot + PO[:, k].astype(np.float64) * normal[:, k].astype(np.float64)
        vc = (dot / dist.astype(np.float64)).astype(F32)
        ratio = np.asarray(max_d, F32) / dist
    rule = np.full(n, RULES.index("in_view"), np.int32)
    checks = [("angle", vc < F32(cos_limit)),
              ("dist_large", dist > maxd), ("dist_small", dist < mind),
              ("v_out", (v < b[2]) | (v > b[3])), ("u_out", (u < b[0]) | (u > b[1])),
              ("behind", Pc[:, 2] < F32(0.0))]
    for name, bad in checks:  # the earliest rule wins: applied last
        rule[bad] = RULES.index(name)
    inv = rule == RULES.index("in_view")
    level = np.zeros(n, np.int32)
    if inv.any():
        level[inv] = predict_scale(np.asarray(max_d, F32)[inv], dist[inv], log_sf, nlevels)
    z = F32(0)
    return dict(in_view=inv.astype(np.uint8), u=np.where(inv, u, z).astype(F32), v=np.where(inv, v, z).astype(F32),
                view_cos=np.where(inv, vc, z).astype(F32), level=level, rule=rule, Pc=Pc, invz=invz, u_raw=u, v_raw=v,
                dist=dist, min_dist=mind, max_dist=maxd, view_cos_raw=vc, ratio=ratio)


def project_last(T, K, bounds4, pos):
    """ORBmatcher.cc:1252-1268: invzc = 1.0 / z in double then float, skip invzc < 0, then the image bounds."""
    T = np.asarray(T, F32)[:3, :4]
    fx, fy, cx, cy = [F32(k) for k in K]
    b = np.asarray(bounds4, F32)
    with np.errstate(all="ignore"):
        Pc = gemm_small(T, pos)
        invz = (1.0 / Pc[:, 2].astype(np.float64)).astype(F32)
        u = fx * Pc[:, 0] * invz + cx
        v = fy * Pc[:, 1] * invz + cy
    ok = ~(invz < 0) & ~((u < b[0]) | (u > b[1])) & ~((v < b[2]) | (v > b[3]))
    z = F32(0)
    return ok.astype(np.uint8), np.where(ok, u, z).astype(F32), np.where(ok, v, z).astype(F32)


def radius_by_viewing_cos(view_cos, th):
    """RadiusByViewingCos (ORBmatcher.cc:123-128) compares the float with the DOUBLE literal 0.998; r *= th only when
    th != 1.0 (:50, :64)."""
    r = np.where(np.asarray(view_cos, F32).astype(np.float64) > 0.998, F32(2.5), F32(4.0)).astype(F32)
    if F32(th) != 1.0:
        r = (r * F32(th)).astype(F32)
    return r


def local_map_query(table, rows, frame_rows, T, K, bounds4, scale_factors, log_sf, nlevels, th):
    """SearchLocalPoints (Tracking.cc:964-1006) as a window query over the local-map list `rows`.
    table: dict of numpy columns pos, normal, min_d, max_d, desc, has_obs, bad.  frame_rows: the table row of each
    keypoint of the current frame or -1.  -> (track dict over the list, query dict for match_window, tgt_blocked,
    n_to_match).  Bad frame points are NULLed first (:970-973), so they are neither stamped as seen nor blocking."""
    rows = np.asarray(rows, np.int64)
    fr = np.asarray(frame_rows, np.int64)
    bad = table["bad"].astype(bool)
    live = fr[(fr >= 0)]
    live = live[~bad[live]]
    seen = np.zeros(len(table["bad"]), bool)
    seen[live] = True
    tr = is_in_frustum(T, K, bounds4, table["pos"][rows], table["normal"][rows], table["min_d"][rows],
                       table["max_d"][rows], log_sf, nlevels, 0.5)
    skip = seen[rows] | bad[rows]
    for k in ("in_view", "u", "v", "view_cos", "level"):
        tr[k] = np.where(skip, 0, tr[k]).astype(tr[k].dtype)
    valid = tr["in_view"].astype(np.uint8)
    lvl = tr["level"]
    sf = np.asarray(scale_factors, F32)
    radius = (radius_by_viewing_cos(tr["view_cos"], th) * sf[lvl]).astype(F32)
    q = dict(desc=table["desc"][rows], u=tr["u"], v=tr["v"], radius=radius, min_level=(lvl - 1).astype(np.int32),
             max_level=lvl.astype(np.int32), valid=valid, blocks=table["has_obs"][rows].astype(np.uint8))
    blocked = np.zeros(len(fr), np.uint8)
    has = fr >= 0
    blocked[has] = (table["has_obs"][fr[has]] != 0) & ~bad[fr[has]]
    return tr, q, blocked, int(valid.sum())


def last_frame_query(table, last_rows, last_octave, last_angle, cur_rows, T, K, bounds4, scale_factors, th):
    """SearchByProjection(cur, last, th, true), ORBmatcher.cc:1223-1354, as a window query over the last frame's
    keypoints.  last_rows: table row of each last-frame keypoint, -1 for NULL or outlier (:1247-1250).  cur_rows: the
    current frame's rows or -1 (a slot whose point has observations is unavailable, :1291-1293)."""
    lr = np.asarray(last_rows, np.int64)
    has = lr >= 0
    r0 = np.where(has, lr, 0)
    ok, u, v = project_last(T, K, bounds4, table["pos"][r0])
    valid = (ok.astype(bool) & has).astype(np.uint8)
    oct_ = np.asarray(last_octave, np.int32)
    sf = np.asarray(scale_factors, F32)
    radius = np.where(valid, F32(th) * sf[np.clip(oct_, 0, len(sf) - 1)], F32(0)).astype(F32)
    z = F32(0)
    q = dict(desc=table["desc"][r0], u=np.where(valid, u, z).astype(F32), v=np.where(valid, v, z).astype(F32),
             radius=radius, min_level=(oct_ - 1).astype(np.int32), max_level=(oct_ + 1).astype(np.int32), valid=valid,
             blocks=table["has_obs"][r0].astype(np.uint8), angle=np.asarray(last_angle, F32))
    cr = np.asarray(cur_rows, np.int64) if cur_rows is not None else None
    blocked = None
    if cr is not None:
        blocked = np.zeros(len(cr), np.uint8)
        blocked[cr >= 0] = table["has_obs"][cr[cr >= 0]] != 0
    return q, blocked
