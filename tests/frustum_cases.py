"""Scenes for the isInFrustum / PredictScale tests: random views at the benchmark's camera and hand-built points that
put each rule of Frame::isInFrustum (Frame.cc:316-375) and each level threshold of MapPoint::PredictScale
(MapPoint.cc:476-485) on its edge.

A scene is a dict: T (3x4 float32 mTcw), K (fx, fy, cx, cy), bounds4 (mnMinX, mnMaxX, mnMinY, mnMaxY), pos, normal
(n x 3), min_d, max_d (mfMinDistance / mfMaxDistance), log_sf, nlevels.  The edge scene uses K = (1, 1, 0, 0) and
T = [I | 0], so that u = X / Z, v = Y / Z and, for points on the optical axis, dist = Z and viewCos = the normal's z
component, all exactly: every edge value is then a float the test picks."""
import numpy as np

F32 = np.float32
K_EUROC = (458.654, 457.296, 367.215, 248.375)
BOUNDS_752 = (0.0, 752.0, 0.0, 480.0)
NLEVELS = 8


def scale_tables(scale_factor=1.2, nlevels=NLEVELS):
    """mvScaleFactors (ORBextractor.cc:345-352, float products) and mfLogScaleFactor = log(float) (Frame.cc:112)."""
    import frustum_ref
    sf = np.ones(nlevels, F32)
    for i in range(1, nlevels):
        sf[i] = sf[i - 1] * F32(scale_factor)
    return sf, F32(frustum_ref.logf(np.array([scale_factor], F32))[0])


SF, LOG_SF = scale_tables()


def up(x, k=1):
    x = F32(x)
    for _ in range(k):
        x = np.nextafter(x, F32(np.inf))
    return F32(x)


def down(x, k=1):
    x = F32(x)
    for _ in range(k):
        x = np.nextafter(x, F32(-np.inf))
    return F32(x)


def small_pose(rng, rot=0.05, trans=0.2):
    w = rng.normal(0, rot, 3)
    th = np.linalg.norm(w)
    k = w / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    R = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx
    T = np.zeros((3, 4), np.float32)
    T[:, :3] = R
    T[:, 3] = rng.normal(0, trans, 3)
    return T


def random_scene(rng, n, K=K_EUROC, bounds4=BOUNDS_752):
    """Points spread over the image and a margin around it, some behind the camera, distances and normals drawn so
    that every rule decides some points."""
    fx, fy, cx, cy = K
    T = small_pose(rng)
    px = rng.uniform(bounds4[0] - 60, bounds4[1] + 60, n)
    py = rng.uniform(bounds4[2] - 60, bounds4[3] + 60, n)
    z = rng.uniform(0.5, 20.0, n) * np.where(rng.random(n) < 0.05, -1, 1)
    pc = np.stack([(px - cx) / fx * z, (py - cy) / fy * z, z], 1)
    R, t = T[:, :3].astype(np.float64), T[:, 3].astype(np.float64)
    pw = ((pc - t) @ R).astype(np.float32)  # R^T (pc - t)
    Ow = -R.T @ t
    d = np.linalg.norm(pw - Ow, axis=1)
    view = (pw - Ow) / d[:, None]
    normal = (view + rng.normal(0, 0.6, (n, 3))).astype(np.float32)
    normal /= np.linalg.norm(normal, axis=1, keepdims=True)
    max_d = (d * rng.uniform(0.7, 6.0, n)).astype(np.float32)
    min_d = (max_d / rng.uniform(2.0, 30.0, n)).astype(np.float32)
    hi = rng.random(n) < 0.05
    min_d[hi] = (d[hi] * rng.uniform(1.0, 1.6, hi.sum())).astype(np.float32)  # too close
    return dict(T=T, K=K, bounds4=bounds4, pos=pw, normal=normal.astype(np.float32), min_d=min_d, max_d=max_d,
                log_sf=LOG_SF, nlevels=NLEVELS)


def thresholds_by_bisection(predict, log_sf=LOG_SF, nlevels=NLEVELS):
    """thr[k - 1] = the largest positive float ratio whose level is below k, found by bisection over float bit
    patterns of ratio = max / 1.0 with `predict(max_d_array, dist_array)` (levels are non-decreasing in the ratio)."""
    out = np.zeros(nlevels - 1, F32)
    for k in range(1, nlevels):
        lo, hi = 0, 0x7F7FFFFF  # level(lo) < k <= level(hi)
        while hi - lo > 1:
            mid = (lo + hi) // 2
            r = np.array([mid], np.uint32).view(F32)
            if predict(r, np.ones(1, F32))[0] < k:
                lo = mid
            else:
                hi = mid
        out[k - 1] = np.array([lo], np.uint32).view(F32)[0]
    return out


def edge_scene(thresholds):
    """One point per edge (see the module docstring).  Returns (scene, names): names[i] says what point i tests."""
    pts = []

    def add(name, P, normal=(0.0, 0.0, 1.0), min_d=0.0, max_d=1e6):
        pts.append((name, [F32(c) for c in P], [F32(c) for c in normal], F32(min_d), F32(max_d)))

    # PcZ = +0 (u = 0 * inf = NaN passes the bounds, dist = 0, viewCos = NaN, ratio = inf), -0 (passes `PcZ < 0`, then
    # u = +inf), -1 ulp (behind)
    add("z=+0", (0.0, 0.0, 0.0))
    add("z=-0", (-0.5, -0.5, -0.0))
    add("z=-1ulp", (0.0, 0.0, down(0.0)))
    # u and v at each bound (inclusive) and one ulp outside; bounds (-1, 1.25, -0.75, 0.5)
    b = (F32(-1.0), F32(1.25), F32(-0.75), F32(0.5))
    add("u=min", (b[0], 0.0, 1.0)); add("u=min-1ulp", (down(b[0]), 0.0, 1.0))
    add("u=max", (b[1], 0.0, 1.0)); add("u=max+1ulp", (up(b[1]), 0.0, 1.0))
    add("v=min", (0.0, b[2], 1.0)); add("v=min-1ulp", (0.0, down(b[2]), 1.0))
    add("v=max", (0.0, b[3], 1.0)); add("v=max+1ulp", (0.0, up(b[3]), 1.0))
    # dist = Z on the axis; minDistance = 0.8f * 1.25, maxDistance = 1.2f * 10
    mn, mx = F32(0.8) * F32(1.25), F32(1.2) * F32(10.0)
    for name, z in (("dist=min", mn), ("dist=min-1ulp", down(mn)), ("dist=min+1ulp", up(mn)),
                    ("dist=max", mx), ("dist=max+1ulp", up(mx)), ("dist=max-1ulp", down(mx))):
        add(name, (0.0, 0.0, z), min_d=1.25, max_d=10.0)
    # viewCos = the normal's z component at Z = 2
    for name, c in (("cos=0.5", F32(0.5)), ("cos=0.5-1ulp", down(0.5)), ("cos=0.998f", F32(0.998)),
                    ("cos=0.998f-1ulp", down(0.998)), ("cos=0.998f+1ulp", up(0.998))):
        s = F32(np.sqrt(max(0.0, 1.0 - float(c) * float(c))))
        add(name, (0.0, 0.0, 2.0), normal=(0.0, s, c))
    # ratio = max_d / 1 at Z = 1: every threshold and one ulp either side, below 1, exactly 1, very large
    for k, t in enumerate(thresholds, 1):
        add(f"ratio=thr{k}", (0.0, 0.0, 1.0), max_d=t)
        add(f"ratio=thr{k}+1ulp", (0.0, 0.0, 1.0), max_d=up(t))
        add(f"ratio=thr{k}-1ulp", (0.0, 0.0, 1.0), max_d=down(t))
    add("ratio=0.9", (0.0, 0.0, 1.0), max_d=0.9)
    add("ratio=1", (0.0, 0.0, 1.0), max_d=1.0)
    add("ratio=1e30", (0.0, 0.0, 1.0), max_d=1e30)
    T = np.zeros((3, 4), np.float32)
    T[:, :3] = np.eye(3)
    T[:, 3] = F32(-0.0)
    names = [p[0] for p in pts]
    scene = dict(T=T, K=(1.0, 1.0, 0.0, 0.0), bounds4=b, pos=np.array([p[1] for p in pts], F32),
                 normal=np.array([p[2] for p in pts], F32), min_d=np.array([p[3] for p in pts], F32),
                 max_d=np.array([p[4] for p in pts], F32), log_sf=LOG_SF, nlevels=NLEVELS)
    return scene, names


def same_bits(a, b):
    """Equal bit patterns, or both NaN (the device's canonical NaN differs from the CPU's)."""
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype.kind != "f":
        return a == b
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
