"""Synthetic tracking scenes for the MapPoint-table tests and tools/localmap_probe.py: a local map seen from a current
camera (tests/frustum_cases.random_scene) and a current frame whose keypoints are noisy projections of part of it, with
the table, resident frame and call arguments built from them."""
import numpy as np

import frustum_cases as FC
import frustum_ref
from swarmmap_b200.matcher import Frame, MapPointTable, ResidentFrame

F32 = np.float32


def _b4_to_frame(b4):
    return (b4[0], b4[2], b4[1], b4[3])  # Frame.bounds = (mnMinX, mnMinY, mnMaxX, mnMaxY)


def make_world(rng, npts, K=FC.K_EUROC, b4=FC.BOUNDS_752, extra=400, frac_seen=0.15, frac_bad=0.03):
    """A local map of npts points seen from a current camera, and a current frame whose keypoints are noisy
    projections of 60 % of them (descriptors a few bits away) plus `extra` unrelated keypoints."""
    sc = FC.random_scene(rng, npts, K, b4)
    n = npts
    tab = dict(pos=sc["pos"], normal=sc["normal"], min_d=sc["min_d"], max_d=sc["max_d"],
               desc=rng.integers(0, 256, (n, 32), dtype=np.uint8), has_obs=(rng.random(n) < 0.9).astype(np.uint8),
               bad=(rng.random(n) < frac_bad).astype(np.uint8))
    tr = frustum_ref.is_in_frustum(sc["T"], K, b4, sc["pos"], sc["normal"], sc["min_d"], sc["max_d"], FC.LOG_SF, 8)
    src = np.nonzero((tr["in_view"] == 1) & (rng.random(n) < 0.6))[0]
    kx = np.clip(tr["u"][src] + rng.normal(0, 1.0, len(src)), b4[0], b4[1] - 0.01)
    ky = np.clip(tr["v"][src] + rng.normal(0, 1.0, len(src)), b4[2], b4[3] - 0.01)
    ko = np.clip(tr["level"][src] - rng.integers(0, 2, len(src)), 0, 7)
    kd = tab["desc"][src].copy()
    flips = rng.integers(0, 256, (len(src), 6))
    for c in range(6):
        kd[np.arange(len(src)), flips[:, c] // 8] ^= (1 << (flips[:, c] % 8)).astype(np.uint8)
    ex = np.stack([rng.uniform(b4[0], b4[1] - 0.01, extra), rng.uniform(b4[2], b4[3] - 0.01, extra)], 1)
    x = np.concatenate([kx, ex[:, 0]]).astype(F32)
    y = np.concatenate([ky, ex[:, 1]]).astype(F32)
    octv = np.concatenate([ko, rng.integers(0, 8, extra)]).astype(np.int32)
    desc = np.concatenate([kd, rng.integers(0, 256, (extra, 32), dtype=np.uint8)])
    ang = rng.uniform(0, 360, len(x)).astype(F32)
    perm = rng.permutation(len(x))
    F = Frame(x[perm], y[perm], octv[perm], ang[perm], desc[perm], _b4_to_frame(b4), FC.SF)
    owner = np.concatenate([src, np.full(extra, -1)])[perm]
    frame_rows = np.where(rng.random(len(x)) < frac_seen, owner, -1).astype(np.int32)
    rows = rng.permutation(n).astype(np.int32)
    return dict(T=sc["T"], K=K, b4=b4, tab=tab, F=F, frame_rows=frame_rows, rows=rows, owner=owner)


def upload_table(tab, table=None, device=0):
    t = table if table is not None else MapPointTable(device)
    n = len(tab["pos"])
    return t.upsert(np.arange(n, dtype=np.int32), tab["pos"], tab["normal"], tab["min_d"], tab["max_d"], tab["desc"],
                    tab["has_obs"], tab["bad"])


def resident(F):
    return ResidentFrame().upload(F)


def points_kw(w, rf, table, th, **kw):
    d = dict(F=rf, table=table, Tcw=w["T"], K=w["K"], log_scale_factor=FC.LOG_SF, rows=w["rows"],
             frame_rows=w["frame_rows"], th=th, scale_factors=FC.SF)
    d.update(kw)
    return d
