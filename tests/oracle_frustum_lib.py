"""ctypes binding of the isInFrustum / PredictScale oracle (oracle/liborb_oracle_frustum.so, oracle/orb_oracle_frustum.cpp).

TEST INFRASTRUCTURE: imported by tests/, __graft_entry__ and tools/ only; the product package never imports it."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
SO = os.path.join(ORACLE_DIR, "liborb_oracle_frustum.so")
SRC = os.path.join(ORACLE_DIR, "orb_oracle_frustum.cpp")
# the flags of oracle/Makefile: no FMA contraction, so the float / double sums round as the reference's do
CXX_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra", "-shared"]

_lib = None
_p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731


def build(force=False):
    if force or not os.path.exists(SO) or os.path.getmtime(SRC) > os.path.getmtime(SO):
        subprocess.run([os.environ.get("CXX", "g++")] + CXX_FLAGS + ["-o", SO, SRC, "-lm"], check=True,
                       capture_output=True)
    return SO


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        vp, ci, cf = C.c_void_p, C.c_int, C.c_float
        L.orc_predict_scale.argtypes = [cf, cf, cf, ci]
        L.orc_predict_scale.restype = ci
        L.orc_predict_scale_many.argtypes = [ci, vp, vp, cf, ci, vp]
        L.orc_is_in_frustum.argtypes = [vp, cf, cf, cf, cf, vp, ci, vp, vp, vp, vp, cf, cf, ci, vp, vp, vp, vp, vp]
        L.orc_project_last.argtypes = [vp, cf, cf, cf, cf, vp, ci, vp, vp, vp, vp]
        _lib = L
    return _lib


def predict_scale(max_distance, dist, log_sf, nlevels):
    """MapPoint::PredictScale per element (arrays of float32)."""
    md = np.ascontiguousarray(np.broadcast_to(np.asarray(max_distance, np.float32), np.shape(dist)), np.float32)
    d = np.ascontiguousarray(dist, np.float32)
    out = np.zeros(d.shape, np.int32)
    lib().orc_predict_scale_many(d.size, _p(md), _p(d), float(np.float32(log_sf)), int(nlevels), _p(out))
    return out


def _f(a, shape=None):
    return np.ascontiguousarray(a, np.float32) if shape is None else np.ascontiguousarray(a, np.float32).reshape(shape)


def is_in_frustum(T, K, bounds4, pos, normal, min_d, max_d, log_sf, nlevels, cos_limit=0.5):
    """Frame::isInFrustum for every point.  T: 3x4 (or 4x4) mTcw; K = (fx, fy, cx, cy); bounds4 = (mnMinX, mnMaxX,
    mnMinY, mnMaxY).  -> dict(in_view, u, v, view_cos, level)."""
    T12 = _f(np.asarray(T, np.float32)[:3, :4], (12,))
    b = _f(bounds4)
    pos, normal = _f(pos, (-1, 3)), _f(normal, (-1, 3))
    n = len(pos)
    mn, mx = _f(min_d), _f(max_d)
    out = dict(in_view=np.zeros(n, np.uint8), u=np.zeros(n, np.float32), v=np.zeros(n, np.float32),
               view_cos=np.zeros(n, np.float32), level=np.zeros(n, np.int32))
    fx, fy, cx, cy = [float(np.float32(k)) for k in K]
    lib().orc_is_in_frustum(_p(T12), fx, fy, cx, cy, _p(b), n, _p(pos), _p(normal), _p(mn), _p(mx),
                            float(np.float32(cos_limit)), float(np.float32(log_sf)), int(nlevels), _p(out["in_view"]),
                            _p(out["u"]), _p(out["v"]), _p(out["view_cos"]), _p(out["level"]))
    return out


def project_last(T, K, bounds4, pos):
    """The projection of SearchByProjection(cur, last, th, true) -> (valid, u, v)."""
    T12 = _f(np.asarray(T, np.float32)[:3, :4], (12,))
    b = _f(bounds4)
    pos = _f(pos, (-1, 3))
    n = len(pos)
    valid, u, v = np.zeros(n, np.uint8), np.zeros(n, np.float32), np.zeros(n, np.float32)
    fx, fy, cx, cy = [float(np.float32(k)) for k in K]
    lib().orc_project_last(_p(T12), fx, fy, cx, cy, _p(b), n, _p(pos), _p(valid), _p(u), _p(v))
    return valid, u, v
