"""Host-side mirror of ORB_SLAM2::ORBmatcher (reference code/include/ORBmatcher.h:37-102) on top of
the C ABI.  The matchers take flat views of the Frame/KeyFrame fields they touch; pointers to
MapPoints never cross the boundary (the C++ wrapper in swarmmap_b200/host/ORBmatcher.h gathers the
same arrays from Frame/KeyFrame/MapPoint objects and scatters the results back).
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import FeatVec, FrameView, SwmError, WindowQuery, check, ptr

__all__ = ["ORBmatcher", "Frame", "FeatureVector", "ResidentFrame", "Camera", "MapPointTable"]

GRID_COLS, GRID_ROWS = 64, 48


class Frame:
    """The slice of ORB_SLAM2::Frame / KeyFrame the matchers read: undistorted keypoints (x, y, octave,
    angle), descriptors (N x 32) and the image bounds mnMinX.. (Frame.cc:486-513)."""

    def __init__(self, x, y, octave, angle, desc, bounds, scale_factors=None):
        self.x = np.ascontiguousarray(x, np.float32)
        self.y = np.ascontiguousarray(y, np.float32)
        self.octave = np.ascontiguousarray(octave, np.int32)
        self.angle = np.ascontiguousarray(angle, np.float32)
        self.desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        self.N = len(self.x)
        assert len(self.y) == self.N and len(self.octave) == self.N and len(self.desc) == self.N
        self.bounds = tuple(float(b) for b in bounds)  # (mnMinX, mnMinY, mnMaxX, mnMaxY)
        self.mvScaleFactors = scale_factors

    @classmethod
    def from_keypoints(cls, kps, desc, width, height, scale_factors=None):
        return cls(kps["x"], kps["y"], kps["octave"], kps["angle"], desc, (0.0, 0.0, float(width), float(height)),
                   scale_factors)

    def view(self):
        b = self.bounds
        return FrameView(self.N, ptr(self.x).value, ptr(self.y).value, ptr(self.octave).value, ptr(self.angle).value,
                         ptr(self.desc).value, b[0], b[1], b[2], b[3])


class Camera:
    """mK + mDistCoef of a Frame (code/src/Frame.cc:60-61), k3 = 0 for four-coefficient settings files."""

    def __init__(self, fx, fy, cx, cy, k1=0.0, k2=0.0, p1=0.0, p2=0.0, k3=0.0):
        self.c = _lib.Camera(fx, fy, cx, cy, k1, k2, p1, p2, k3)

    def bounds(self, cols, rows, device=0):
        """Frame::ComputeImageBounds (Frame.cc:486-514): (mnMinX, mnMaxX, mnMinY, mnMaxY), computed on the device."""
        out = np.zeros(4, np.float32)
        rc = _lib.load().swm_camera_bounds(device, C.byref(self.c), int(cols), int(rows), _lib.ptr(out))
        if rc != 0:
            raise _lib.SwmError(f"swm_camera_bounds: {_lib.ERRORS.get(rc, rc)}")
        return out


class ResidentFrame:
    """A Frame whose undistorted keypoints, descriptors and grid live on the device (SURVEY section 8(f) rank 1):
    built straight from the extractor's device output (Frame::UndistortKeyPoints + AssignFeaturesToGrid, Frame.cc:
    454-484, 277-292) or uploaded once from host arrays, then passed to the ORBmatcher methods in place of a Frame."""

    def __init__(self, device=0):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        self.mvScaleFactors = None  # set by from_extractor / upload (the SearchByProjection wrappers read it)
        rc = self._lib.swm_frame_create(device, C.byref(self._h))
        if rc != 0:
            msg = self._lib.swm_frame_last_error(None)
            raise _lib.SwmError(f"swm_frame_create: {_lib.ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")

    def close(self):
        if getattr(self, "_h", None):
            self._lib.swm_frame_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            msg = self._lib.swm_frame_last_error(self._h)
            raise _lib.SwmError(f"{what}: {_lib.ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")

    @property
    def N(self):
        return int(self._lib.swm_frame_size(self._h))

    def from_extractor(self, extractor, index, camera, bounds):
        """Frame `index` of the extractor's last batch; camera may be None (no distortion)."""
        b = np.ascontiguousarray(bounds, np.float32)
        cam = C.byref(camera.c) if camera is not None else None
        self._check(self._lib.swm_frame_from_extractor(self._h, extractor._h, int(index), cam, _lib.ptr(b)),
                    "swm_frame_from_extractor")
        self.mvScaleFactors = extractor.GetScaleFactors()
        return self

    def upload(self, frame):
        v = frame.view()
        self._check(self._lib.swm_frame_upload(self._h, C.byref(v)), "swm_frame_upload")
        self.mvScaleFactors = frame.mvScaleFactors
        return self

    def export_slab(self):
        """The frame as a binary keyframe-feature slab (bytes): header + x, y, octave, angle, descriptors."""
        nbytes = int(self._lib.swm_frame_slab_bytes(self.N))
        buf = np.zeros(nbytes, np.uint8)
        got = C.c_size_t(0)
        self._check(self._lib.swm_frame_export(self._h, _lib.ptr(buf), nbytes, C.byref(got)), "swm_frame_export")
        return buf[:got.value].tobytes()

    def import_slab(self, blob):
        buf = np.frombuffer(blob, np.uint8)
        self._check(self._lib.swm_frame_import(self._h, _lib.ptr(buf), len(buf)), "swm_frame_import")
        return self

    def download(self, grid=False):
        n = self.N
        x = np.zeros(n, np.float32); y = np.zeros(n, np.float32)
        octave = np.zeros(n, np.int32); angle = np.zeros(n, np.float32)
        desc = np.zeros((n, 32), np.uint8)
        starts = np.zeros(64 * 48 + 1, np.int32) if grid else None
        items = np.zeros(max(n, 1), np.int32) if grid else None
        self._check(self._lib.swm_frame_download(self._h, _lib.ptr(x), _lib.ptr(y), _lib.ptr(octave), _lib.ptr(angle),
                                                 _lib.ptr(desc), _lib.ptr(starts) if grid else None,
                                                 _lib.ptr(items) if grid else None), "swm_frame_download")
        out = dict(x=x, y=y, octave=octave, angle=angle, desc=desc)
        if grid:
            out["starts"] = starts
            out["items"] = items[:starts[-1]]
        return out


class FeatureVector:
    """DBoW2::FeatureVector as CSR: ascending node ids, ascending feature indices per node
    (Thirdparty/DBoW2/DBoW2/FeatureVector.cpp:31-45)."""

    def __init__(self, node_of_feature):
        node_of_feature = np.asarray(node_of_feature, np.int64)
        keep = np.nonzero(node_of_feature >= 0)[0]
        order = keep[np.argsort(node_of_feature[keep], kind="stable")]
        nodes = node_of_feature[order]
        self.node_ids, first = np.unique(nodes, return_index=True)
        self.node_ids = self.node_ids.astype(np.uint32)
        self.offsets = np.append(first, len(nodes)).astype(np.int32)
        self.feats = order.astype(np.uint32)

    def view(self):
        return FeatVec(len(self.node_ids), ptr(self.node_ids).value, ptr(self.offsets).value, ptr(self.feats).value)


class ORBmatcher:
    """ORBmatcher(nnratio=0.6, checkOri=true), ORBmatcher.cc:41."""

    TH_HIGH, TH_LOW, HISTO_LENGTH = 100, 50, 30  # ORBmatcher.cc:37-39

    def __init__(self, nnratio=0.6, checkOri=True, device=0):
        self._lib = _lib.load()
        self.mfNNratio = float(nnratio)
        self.mbCheckOrientation = bool(checkOri)
        self.device = int(device)
        h = C.c_void_p()
        rc = self._lib.swm_matcher_create(self.device, C.byref(h))
        if rc != 0:
            raise SwmError(f"swm_matcher_create: {_lib.ERRORS.get(rc, rc)}: "
                           f"{self._lib.swm_matcher_last_error(None).decode()}")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.swm_matcher_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise SwmError(f"{what}: {_lib.ERRORS.get(rc, rc)}: {self._lib.swm_matcher_last_error(self._h).decode()}")

    # ---- DescriptorDistance (ORBmatcher.cc:1511-1525), batched
    def DescriptorDistance(self, a, b):
        a = np.ascontiguousarray(a, np.uint8).reshape(-1, 32)
        b = np.ascontiguousarray(b, np.uint8).reshape(-1, 32)
        assert len(a) == len(b)
        out = np.zeros(len(a), np.int32)
        rc = self._lib.swm_hamming_pairs(ptr(a), ptr(b), len(a), ptr(out), self.device)
        self._check(rc, "swm_hamming_pairs")
        return int(out[0]) if len(out) == 1 else out

    def distance_matrix(self, a, b):
        a = np.ascontiguousarray(a, np.uint8).reshape(-1, 32)
        b = np.ascontiguousarray(b, np.uint8).reshape(-1, 32)
        out = np.zeros((len(a), len(b)), np.uint16)
        self._check(self._lib.swm_hamming_matrix(ptr(a), len(a), ptr(b), len(b), ptr(out), self.device),
                    "swm_hamming_matrix")
        return out

    # ---- the search loop of Fuse (ORBmatcher.cc:824-870, :962-999) and SearchBySim3 (:1098-1134, :1178-1214)
    def window_best(self, tgt, desc, u, v, radius, pred_level, valid, inv_level_sigma2=None, chi2=0.0):
        """Per query: the keypoint of `tgt` inside the window at levels [pred - 1, pred] with the smallest distance
        (first in GetFeaturesInArea order on ties); chi2 > 0 adds Fuse's reprojection gate.  Returns (best_idx,
        best_dist) with -1 / 256 for rows without a surviving candidate; the caller applies TH_LOW / TH_HIGH."""
        from ._lib import BestQuery
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        pl = np.ascontiguousarray(pred_level, np.int32)
        a = dict(u=np.ascontiguousarray(u, np.float32), v=np.ascontiguousarray(v, np.float32),
                 radius=np.ascontiguousarray(radius, np.float32), lo=np.ascontiguousarray(pl - 1, np.int32), hi=pl,
                 valid=np.ascontiguousarray(valid, np.uint8))
        s2 = np.ascontiguousarray(inv_level_sigma2, np.float32) if inv_level_sigma2 is not None else None
        q = BestQuery(len(pl), ptr(desc).value, ptr(a["u"]).value, ptr(a["v"]).value, ptr(a["radius"]).value,
                      ptr(a["lo"]).value, ptr(a["hi"]).value, ptr(a["valid"]).value,
                      ptr(s2).value if s2 is not None else None, len(s2) if s2 is not None else 0, float(chi2))
        bi = np.full(len(pl), -1, np.int32)
        bd = np.full(len(pl), 256, np.int32)
        if isinstance(tgt, ResidentFrame):
            rc = self._lib.swm_window_best_resident(self._h, tgt._h, C.byref(q), ptr(bi), ptr(bd))
        else:
            tv = tgt.view()
            rc = self._lib.swm_window_best(self._h, C.byref(tv), C.byref(q), ptr(bi), ptr(bd))
        self._check(rc, "swm_window_best")
        return bi, bd

    # ---- MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:361-391), batched over MapPoints
    def ComputeDistinctiveDescriptors(self, desc, offsets):
        """desc: (total, 32) observed descriptors, point p owns rows offsets[p]:offsets[p+1].  Returns (best index
        inside each point, its median distance)."""
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        offsets = np.ascontiguousarray(offsets, np.int32)
        npts = len(offsets) - 1
        best = np.full(npts, -1, np.int32)
        med = np.full(npts, -1, np.int32)
        rc = self._lib.swm_distinctive_descriptors(ptr(desc), ptr(offsets), npts, ptr(best), ptr(med), self.device)
        self._check(rc, "swm_distinctive_descriptors")
        return best, med

    # ---- Frame grid (Frame.cc:277-292)
    def grid(self, frame):
        starts = np.zeros(GRID_COLS * GRID_ROWS + 1, np.int32)
        items = np.zeros(max(frame.N, 1), np.int32)
        v = frame.view()
        self._check(self._lib.swm_grid_build(self._h, C.byref(v), ptr(starts), ptr(items)), "swm_grid_build")
        return starts, items[:starts[-1]]

    # ---- SearchForInitialization (ORBmatcher.cc:375-479)
    def SearchForInitialization(self, F1, F2, vbPrevMatched, windowSize=10):
        """vbPrevMatched: (N1, 2) float32, updated in place.  Returns (nmatches, vnMatches12)."""
        assert vbPrevMatched.dtype == np.float32 and vbPrevMatched.shape == (F1.N, 2) and vbPrevMatched.flags.c_contiguous
        matches = np.full(F1.N, -1, np.int32)
        n = C.c_int(0)
        if isinstance(F1, ResidentFrame) != isinstance(F2, ResidentFrame):
            raise TypeError("both frames must be resident or both host-side")
        if isinstance(F1, ResidentFrame):
            rc = self._lib.swm_match_init_resident(self._h, F1._h, F2._h, ptr(vbPrevMatched), ptr(matches),
                                                   int(windowSize), self.mfNNratio, int(self.mbCheckOrientation),
                                                   C.byref(n))
        else:
            v1, v2 = F1.view(), F2.view()
            rc = self._lib.swm_match_init(self._h, C.byref(v1), C.byref(v2), ptr(vbPrevMatched), ptr(matches),
                                          int(windowSize), self.mfNNratio, int(self.mbCheckOrientation), C.byref(n))
        self._check(rc, "swm_match_init")
        return n.value, matches

    # ---- generic windowed projection matcher behind the SearchByProjection overloads
    def match_window(self, tgt, desc, u, v, radius, min_level, max_level, valid, blocks, th_dist, ratio_mode=0,
                     angle=None, tgt_blocked=None, assignment=None, check_ori=None):
        m = len(u)
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        arrs = dict(u=np.ascontiguousarray(u, np.float32), v=np.ascontiguousarray(v, np.float32),
                    radius=np.ascontiguousarray(radius, np.float32),
                    min_level=np.ascontiguousarray(min_level, np.int32),
                    max_level=np.ascontiguousarray(max_level, np.int32),
                    valid=np.ascontiguousarray(valid, np.uint8), blocks=np.ascontiguousarray(blocks, np.uint8))
        check_ori = self.mbCheckOrientation if check_ori is None else bool(check_ori)
        ang = np.ascontiguousarray(angle, np.float32) if angle is not None else None
        if check_ori and ang is None:
            raise ValueError("angle is required when the orientation check is on")
        q = WindowQuery(m, ptr(desc).value, ptr(arrs["u"]).value, ptr(arrs["v"]).value, ptr(arrs["radius"]).value,
                        ptr(arrs["min_level"]).value, ptr(arrs["max_level"]).value, ptr(arrs["valid"]).value,
                        ptr(ang).value if ang is not None else None, ptr(arrs["blocks"]).value)
        if assignment is None:
            assignment = np.full(tgt.N, -1, np.int32)
        tb = np.ascontiguousarray(tgt_blocked, np.uint8) if tgt_blocked is not None else None
        n = C.c_int(0)
        if isinstance(tgt, ResidentFrame):
            rc = self._lib.swm_match_window_resident(self._h, tgt._h, C.byref(q), ptr(tb) if tb is not None else None,
                                                     int(th_dist), int(ratio_mode), self.mfNNratio, int(check_ori),
                                                     ptr(assignment), C.byref(n))
        else:
            tv = tgt.view()
            rc = self._lib.swm_match_window(self._h, C.byref(tv), C.byref(q), ptr(tb) if tb is not None else None,
                                            int(th_dist), int(ratio_mode), self.mfNNratio, int(check_ori),
                                            ptr(assignment), C.byref(n))
        self._check(rc, "swm_match_window")
        return n.value, assignment

    def SearchByProjectionLastFrame(self, cur, last, proj_u, proj_v, valid, th, last_obs_positive=None,
                                    cur_blocked=None):
        """SearchByProjection(Frame &cur, const Frame &last, th, bMono=true), ORBmatcher.cc:1223-1354.
        proj_u/v: last-frame MapPoints projected with cur.mTcw (done by the caller); valid[i] = the point
        exists, is an inlier, has positive depth and projects inside the image."""
        sf = np.asarray(cur.mvScaleFactors, np.float32)
        radius = np.float32(th) * sf[last.octave]
        blocks = np.ones(last.N, np.uint8) if last_obs_positive is None else last_obs_positive
        return self.match_window(cur, last.desc, proj_u, proj_v, radius, last.octave - 1, last.octave + 1, valid,
                                 blocks, self.TH_HIGH, 0, last.angle, cur_blocked)

    def SearchByProjectionMapPoints(self, F, desc, proj_u, proj_v, pred_level, view_cos, valid, th=1.0,
                                    obs_positive=None, blocked=None):
        """SearchByProjection(Frame &F, const vector<MapPoint*>&, th), ORBmatcher.cc:44-121."""
        sf = np.asarray(F.mvScaleFactors, np.float32)
        pred_level = np.asarray(pred_level, np.int32)
        # RadiusByViewingCos (:123-128) compares the float against the DOUBLE literal 0.998
        r = np.where(np.asarray(view_cos, np.float32).astype(np.float64) > 0.998, np.float32(2.5), np.float32(4.0))
        if th != 1.0:
            r = (r * np.float32(th)).astype(np.float32)
        radius = (r.astype(np.float32) * sf[pred_level]).astype(np.float32)
        blocks = np.ones(len(proj_u), np.uint8) if obs_positive is None else obs_positive
        return self.match_window(F, desc, proj_u, proj_v, radius, pred_level - 1, pred_level, valid, blocks,
                                 self.TH_HIGH, 1, None, blocked, check_ori=False)

    def SearchByProjectionKeyFrame(self, cur, kf_desc, kf_angle, proj_u, proj_v, pred_level, valid, th, ORBdist,
                                   cur_has_mappoint=None):
        """SearchByProjection(Frame&, KeyFrame*, sAlreadyFound, th, ORBdist, bGlobal) (relocalisation),
        ORBmatcher.cc:1356-1473.  valid[i]: the KeyFrame MapPoint exists, is good, is not in sAlreadyFound,
        projects inside the image and its distance is inside the scale-invariance range (caller-side checks
        :1380-1407); pred_level = PredictScale.  Any already-assigned slot of `cur` is unavailable (:1413)."""
        sf = np.asarray(cur.mvScaleFactors, np.float32)
        pred_level = np.asarray(pred_level, np.int32)
        radius = (np.float32(th) * sf[pred_level]).astype(np.float32)
        ones = np.ones(len(proj_u), np.uint8)
        return self.match_window(cur, kf_desc, proj_u, proj_v, radius, pred_level - 1, pred_level + 1, valid, ones,
                                 int(ORBdist), 0, kf_angle, cur_has_mappoint)

    def SearchByProjectionSim3(self, kf, desc, proj_u, proj_v, pred_level, valid, th, already_matched=None):
        """SearchByProjection(KeyFrame*, Scw, vpPoints, vpMatched, th) (loop closing), ORBmatcher.cc:264-373.
        valid[i]: the point is good, not already found, in front of the camera, inside the image, inside its
        distance range and within 60 degrees of its normal (caller-side checks :289-329).  The level filter
        [pred-1, pred] of :349-352 is applied inside the window query; no ratio test, no orientation check."""
        sf = np.asarray(kf.mvScaleFactors, np.float32)
        pred_level = np.asarray(pred_level, np.int32)
        radius = (np.float32(th) * sf[pred_level]).astype(np.float32)
        ones = np.ones(len(proj_u), np.uint8)
        return self.match_window(kf, desc, proj_u, proj_v, radius, pred_level - 1, pred_level, valid, ones,
                                 self.TH_LOW, 0, None, already_matched, check_ori=False)

    # ---- SearchByBoW (ORBmatcher.cc:150-262 KeyFrame->Frame, :481-597 KeyFrame<->KeyFrame)
    def SearchByBoW(self, KF, fvKF, validKF, F, fvF, validF=None):
        mode = 0 if validF is None else 1
        validKF = np.ascontiguousarray(validKF, np.uint8)
        v2 = np.ascontiguousarray(validF, np.uint8) if validF is not None else None
        out = np.full(F.N if mode == 0 else KF.N, -1, np.int32)
        n = C.c_int(0)
        fa, fb = fvKF.view(), fvF.view()
        if isinstance(KF, ResidentFrame) != isinstance(F, ResidentFrame):
            raise TypeError("both frames must be resident or both host-side")
        if isinstance(KF, ResidentFrame):
            rc = self._lib.swm_match_bow_resident(self._h, KF._h, C.byref(fa), ptr(validKF), F._h, C.byref(fb),
                                                  ptr(v2) if v2 is not None else None, mode, self.mfNNratio,
                                                  int(self.mbCheckOrientation), ptr(out), C.byref(n))
        else:
            a, b = KF.view(), F.view()
            rc = self._lib.swm_match_bow(self._h, C.byref(a), C.byref(fa), ptr(validKF), C.byref(b), C.byref(fb),
                                         ptr(v2) if v2 is not None else None, mode, self.mfNNratio,
                                         int(self.mbCheckOrientation), ptr(out), C.byref(n))
        self._check(rc, "swm_match_bow")
        return n.value, out


# ---- batched (throughput) forms: P independent problems per call, same results as the single calls

def _frame_fields(fr, keep):
    """(host view pointer, resident handle) of a Frame / ResidentFrame for a batch job."""
    if isinstance(fr, ResidentFrame):
        return None, fr._h
    v = fr.view()
    keep.append(v)
    return C.addressof(v), None


def _window_job(self, keep, tgt, desc, u, v, radius, min_level, max_level, valid, blocks, th_dist, ratio_mode=0,
                angle=None, tgt_blocked=None, assignment=None, check_ori=None):
    from ._lib import WindowJob
    desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
    a = [np.ascontiguousarray(u, np.float32), np.ascontiguousarray(v, np.float32),
         np.ascontiguousarray(radius, np.float32), np.ascontiguousarray(min_level, np.int32),
         np.ascontiguousarray(max_level, np.int32), np.ascontiguousarray(valid, np.uint8),
         np.ascontiguousarray(blocks, np.uint8)]
    check_ori = self.mbCheckOrientation if check_ori is None else bool(check_ori)
    ang = np.ascontiguousarray(angle, np.float32) if angle is not None else None
    if check_ori and ang is None:
        raise ValueError("angle is required when the orientation check is on")
    q = WindowQuery(len(a[0]), ptr(desc).value, ptr(a[0]).value, ptr(a[1]).value, ptr(a[2]).value, ptr(a[3]).value,
                    ptr(a[4]).value, ptr(a[5]).value, ptr(ang).value if ang is not None else None, ptr(a[6]).value)
    asg = np.full(tgt.N, -1, np.int32) if assignment is None else assignment
    tb = np.ascontiguousarray(tgt_blocked, np.uint8) if tgt_blocked is not None else None
    hv, hr = _frame_fields(tgt, keep)
    keep.extend([desc, a, ang, q, tb, asg])
    return WindowJob(hv, hr, C.addressof(q), ptr(tb).value if tb is not None else None, int(th_dist), int(ratio_mode),
                     self.mfNNratio, int(check_ori), ptr(asg).value, 0), asg


def _match_window_batch(self, jobs):
    """jobs: list of dicts with match_window's arguments.  Returns [(nmatches, assignment), ...]."""
    from ._lib import WindowJob
    keep, outs = [], []
    arr = (WindowJob * len(jobs))()
    for i, kw in enumerate(jobs):
        arr[i], asg = _window_job(self, keep, **kw)
        outs.append(asg)
    self._check(self._lib.swm_match_window_batch(self._h, arr, len(jobs)), "swm_match_window_batch")
    return [(int(arr[i].nmatches), outs[i]) for i in range(len(jobs))]


def _search_for_initialization_batch(self, pairs, windowSize=10):
    """pairs: list of (F1, F2, vbPrevMatched (N1 x 2 float32, updated in place)).  Returns [(nmatches, vnMatches12)]."""
    from ._lib import InitJob
    keep, outs = [], []
    arr = (InitJob * len(pairs))()
    for i, (F1, F2, prev) in enumerate(pairs):
        assert prev.dtype == np.float32 and prev.shape == (F1.N, 2) and prev.flags.c_contiguous
        if isinstance(F1, ResidentFrame) != isinstance(F2, ResidentFrame):
            raise TypeError("both frames must be resident or both host-side")
        m12 = np.full(F1.N, -1, np.int32)
        v1, r1 = _frame_fields(F1, keep)
        v2, r2 = _frame_fields(F2, keep)
        arr[i] = InitJob(v1, v2, r1, r2, ptr(prev).value, ptr(m12).value, int(windowSize), self.mfNNratio,
                         int(self.mbCheckOrientation), 0)
        outs.append(m12)
    self._check(self._lib.swm_match_init_batch(self._h, arr, len(pairs)), "swm_match_init_batch")
    return [(int(arr[i].nmatches), outs[i]) for i in range(len(pairs))]


def _search_by_bow_batch(self, jobs):
    """jobs: list of (KF, fvKF, validKF, F, fvF, validF-or-None).  Returns [(nmatches, matches)]."""
    from ._lib import BowJob
    keep, outs = [], []
    arr = (BowJob * len(jobs))()
    for i, (KF, fvKF, validKF, F, fvF, validF) in enumerate(jobs):
        mode = 0 if validF is None else 1
        if isinstance(KF, ResidentFrame) != isinstance(F, ResidentFrame):
            raise TypeError("both frames must be resident or both host-side")
        v1 = np.ascontiguousarray(validKF, np.uint8)
        v2 = np.ascontiguousarray(validF, np.uint8) if validF is not None else None
        out = np.full(F.N if mode == 0 else KF.N, -1, np.int32)
        fa, fb = fvKF.view(), fvF.view()
        h1, r1 = _frame_fields(KF, keep)
        h2, r2 = _frame_fields(F, keep)
        keep.extend([v1, v2, fa, fb])
        arr[i] = BowJob(h1, h2, r1, r2, C.addressof(fa), C.addressof(fb), ptr(v1).value,
                        ptr(v2).value if v2 is not None else None, mode, self.mfNNratio, int(self.mbCheckOrientation),
                        ptr(out).value, 0)
        outs.append(out)
    self._check(self._lib.swm_match_bow_batch(self._h, arr, len(jobs)), "swm_match_bow_batch")
    return [(int(arr[i].nmatches), outs[i]) for i in range(len(jobs))]


ORBmatcher.match_window_batch = _match_window_batch
ORBmatcher.SearchForInitializationBatch = _search_for_initialization_batch
ORBmatcher.SearchByBoWBatch = _search_by_bow_batch


def resident_frames_from_extractor(extractor, count, camera, bounds, device=0, frames=None):
    """ResidentFrames for frames 0..count-1 of the extractor's last batch (two launches, one count read-back)."""
    lib = _lib.load()
    frames = frames if frames is not None else [ResidentFrame(device) for _ in range(count)]
    hs = (C.c_void_p * count)(*[f._h for f in frames[:count]])
    b = np.ascontiguousarray(bounds, np.float32)
    cam = C.byref(camera.c) if camera is not None else None
    rc = lib.swm_frames_from_extractor(hs, count, extractor._h, None, cam, _lib.ptr(b))
    frames[0]._check(rc, "swm_frames_from_extractor")
    sf = extractor.GetScaleFactors()
    for f in frames[:count]:
        f.mvScaleFactors = sf
    return frames


def _search_for_triangulation(self, KF1, fv1, no_mp1, KF2, fv2, no_mp2, F12, ex, ey, scale_factors2, level_sigma2):
    """SearchForTriangulation(pKF1, pKF2, F12, vMatchedPairs, bOnlyStereo=false), ORBmatcher.cc:599-749 (monocular).
    no_mp1 / no_mp2: 1 where the keypoint has no MapPoint yet; (ex, ey): epipole of KF1's centre in KF2 (:605-611).
    Returns (nmatches, vMatches12); vMatchedPairs = [(i, m) for i, m in enumerate(vMatches12) if m >= 0]."""
    from ._lib import TriangulationQuery
    v1 = np.ascontiguousarray(no_mp1, np.uint8)
    v2 = np.ascontiguousarray(no_mp2, np.uint8)
    F = np.ascontiguousarray(F12, np.float32).reshape(9)
    sf = np.ascontiguousarray(scale_factors2, np.float32)
    s2 = np.ascontiguousarray(level_sigma2, np.float32)
    q = TriangulationQuery(ptr(F).value, float(ex), float(ey), ptr(sf).value, ptr(s2).value, len(sf))
    out = np.full(KF1.N, -1, np.int32)
    n = C.c_int(0)
    fa, fb = fv1.view(), fv2.view()
    if isinstance(KF1, ResidentFrame) != isinstance(KF2, ResidentFrame):
        raise TypeError("both keyframes must be resident or both host-side")
    if isinstance(KF1, ResidentFrame):
        rc = self._lib.swm_match_triangulation_resident(self._h, KF1._h, C.byref(fa), ptr(v1), KF2._h, C.byref(fb), ptr(v2),
                                                        C.byref(q), int(self.mbCheckOrientation), ptr(out), C.byref(n))
    else:
        a, b = KF1.view(), KF2.view()
        rc = self._lib.swm_match_triangulation(self._h, C.byref(a), C.byref(fa), ptr(v1), C.byref(b), C.byref(fb), ptr(v2),
                                               C.byref(q), int(self.mbCheckOrientation), ptr(out), C.byref(n))
    self._check(rc, "swm_match_triangulation")
    return n.value, out


ORBmatcher.SearchForTriangulation = _search_for_triangulation


class MapPointTable:
    """MapPoints resident on one device (world position, normal, mfMinDistance / mfMaxDistance, descriptor,
    Observations() > 0, bad flag), one row each, for the tracking projections ORBmatcher.search_local_map /
    search_last_frame.  Rows are the caller's: LocalMapping rewrites a point with upsert when it changes, and a query
    uploads only row indices and the pose.  An upsert never overtakes a query still reading the table, and a query
    sees every upsert issued before it."""

    def __init__(self, device=0, capacity=0):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        rc = self._lib.swm_mappoints_create(int(device), int(capacity), C.byref(self._h))
        if rc != 0:
            msg = self._lib.swm_mappoints_last_error(None)
            raise SwmError(f"swm_mappoints_create: {_lib.ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")

    def close(self):
        if getattr(self, "_h", None):
            self._lib.swm_mappoints_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def size(self):
        return int(self._lib.swm_mappoints_size(self._h))

    def upsert(self, rows, pos, normal, min_d, max_d, desc, has_obs, bad=None):
        """Writes rows (a row given twice takes its last entry); pos / normal (n, 3), desc (n, 32)."""
        rows = np.ascontiguousarray(rows, np.int32).reshape(-1)
        n = len(rows)
        a = [np.ascontiguousarray(pos, np.float32).reshape(n, 3), np.ascontiguousarray(normal, np.float32).reshape(n, 3),
             np.ascontiguousarray(min_d, np.float32).reshape(n), np.ascontiguousarray(max_d, np.float32).reshape(n),
             np.ascontiguousarray(desc, np.uint8).reshape(n, 32), np.ascontiguousarray(has_obs, np.uint8).reshape(n),
             np.ascontiguousarray(np.zeros(n, np.uint8) if bad is None else bad, np.uint8).reshape(n)]
        rc = self._lib.swm_mappoints_upsert(self._h, n, ptr(rows), *[ptr(x) for x in a])
        if rc != 0:
            raise SwmError(f"swm_mappoints_upsert: {_lib.ERRORS.get(rc, rc)}: "
                           f"{self._lib.swm_mappoints_last_error(self._h).decode()}")
        return self


def _projection(Tcw, K, scale_factors, log_scale_factor):
    T = np.ascontiguousarray(np.asarray(Tcw, np.float32)[:3, :4]).reshape(12)
    sf = np.ascontiguousarray(scale_factors, np.float32)
    p = _lib.Projection((C.c_float * 12)(*[float(x) for x in T]), *[float(np.float32(k)) for k in K], ptr(sf).value,
                        float(np.float32(log_scale_factor)), len(sf))
    return p, sf


def _localmap_job(self, keep, mode, F, table, Tcw, K, log_scale_factor, rows, frame_rows=None, th=1.0, last=None,
                  scale_factors=None, track=True, assignment=None):
    """One swm_localmap_job.  Returns (job, outputs dict)."""
    if not isinstance(F, ResidentFrame) or (last is not None and not isinstance(last, ResidentFrame)):
        raise TypeError("the tracking projections take resident frames")
    sf = F.mvScaleFactors if scale_factors is None else scale_factors
    proj, sfa = _projection(Tcw, K, sf, log_scale_factor)
    rows = np.ascontiguousarray(rows, np.int32).reshape(-1)
    fr = np.ascontiguousarray(frame_rows, np.int32).reshape(-1) if frame_rows is not None else None
    if fr is not None and len(fr) != F.N:  # the library reads one entry per keypoint
        raise ValueError(f"frame_rows has {len(fr)} entries, the frame {F.N} keypoints")
    if mode == _lib.LOCALMAP_LAST and (last is None or len(rows) != last.N):
        raise ValueError("the last-frame projection takes one row per keypoint of `last`")
    out = dict(assignment=np.full(F.N, -1 if mode == _lib.LOCALMAP_POINTS else -3, np.int32)
               if assignment is None else assignment)
    tr = None
    if mode == _lib.LOCALMAP_POINTS and track:
        m = len(rows)
        out["track"] = dict(in_view=np.zeros(m, np.uint8), u=np.zeros(m, np.float32), v=np.zeros(m, np.float32),
                            view_cos=np.zeros(m, np.float32), level=np.zeros(m, np.int32))
        t = out["track"]
        tr = _lib.TrackOut(ptr(t["in_view"]).value, ptr(t["u"]).value, ptr(t["v"]).value, ptr(t["view_cos"]).value,
                           ptr(t["level"]).value)
    keep.extend([proj, sfa, rows, fr, tr, out])
    job = _lib.LocalMapJob(mode, F._h, table._h, C.addressof(proj), ptr(rows).value, len(rows),
                           last._h if last is not None else None, ptr(fr).value if fr is not None else None, float(th),
                           self.mfNNratio, int(self.mbCheckOrientation), C.addressof(tr) if tr is not None else None,
                           ptr(out["assignment"]).value, 0, 0)
    return job, out


def _search_local_map(self, F, table, Tcw, K, log_scale_factor, rows, frame_rows=None, th=1.0, scale_factors=None,
                      track=True):
    """Tracking::SearchLocalPoints (Tracking.cc:964-1006) on the device: the MapPoints of the local map (table rows
    in list order) that the current frame does not hold already and that pass isInFrustum(pMP, 0.5) are matched into
    F with SearchByProjection(F, vpMapPoints, th).  frame_rows: the table row of each keypoint of F or -1.
    Returns (nmatches, assignment = list index per keypoint or -1, n_to_match, tracking fields of the list or None)."""
    r = _search_local_map_batch(self, [dict(F=F, table=table, Tcw=Tcw, K=K, log_scale_factor=log_scale_factor, rows=rows,
                                            frame_rows=frame_rows, th=th, scale_factors=scale_factors, track=track)])
    return r[0]


def _search_last_frame(self, cur, last, table, Tcw, K, log_scale_factor, last_rows, cur_rows=None, th=15.0,
                       scale_factors=None, assignment=None):
    """SearchByProjection(cur, last, th, bMono = true), ORBmatcher.cc:1223-1354, from the table.  last_rows: the table
    row of each keypoint of `last`, -1 for NULL or outlier.  assignment (in/out, default -3 = untouched): the
    last-frame keypoint matched at each slot of cur, -1 where the rotation check pruned it.  Returns (nmatches,
    assignment)."""
    r = _search_local_map_batch(self, [dict(mode=_lib.LOCALMAP_LAST, F=cur, last=last, table=table, Tcw=Tcw, K=K,
                                            log_scale_factor=log_scale_factor, rows=last_rows, frame_rows=cur_rows, th=th,
                                            scale_factors=scale_factors, assignment=assignment)])
    return r[0][0], r[0][1]


def _search_local_map_batch(self, jobs):
    """jobs: dicts with search_local_map's arguments (mode LOCALMAP_POINTS, the default) or search_last_frame's
    (mode LOCALMAP_LAST, with F = cur and rows = last_rows).  One upload, seven launches, one download.
    Returns [(nmatches, assignment, n_to_match, track-or-None)]."""
    keep, outs = [], []
    arr = (_lib.LocalMapJob * len(jobs))()
    for i, kw in enumerate(jobs):
        kw = dict(kw)
        mode = kw.pop("mode", _lib.LOCALMAP_POINTS)
        arr[i], out = _localmap_job(self, keep, mode, **kw)
        outs.append(out)
    self._check(self._lib.swm_match_local_map_batch(self._h, arr, len(jobs)), "swm_match_local_map_batch")
    return [(int(arr[i].nmatches), outs[i]["assignment"], int(arr[i].n_to_match), outs[i].get("track"))
            for i in range(len(jobs))]


ORBmatcher.search_local_map = _search_local_map
ORBmatcher.search_last_frame = _search_last_frame
ORBmatcher.search_local_map_batch = _search_local_map_batch


def smoke(kps, desc):
    """Tiny matcher call for __graft_entry__.smoke(): match a frame against itself."""
    f = Frame.from_keypoints(kps, desc, 752, 480)
    m = ORBmatcher(0.9, True)
    prev = np.stack([f.x, f.y], 1).astype(np.float32).copy()
    n, m12 = m.SearchForInitialization(f, f, prev, 100)
    lvl0 = int((f.octave == 0).sum())
    assert n > 0.5 * lvl0, (n, lvl0)
    ok = m12[m12 >= 0] == np.nonzero(m12 >= 0)[0]
    assert ok.mean() > 0.95
    print(f"matcher smoke ok: {n} self-matches of {lvl0} level-0 keypoints")
