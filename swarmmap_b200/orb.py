"""Host-side mirror of the reference's ORB front-end classes, on top of the C ABI (libswm_orb.so).

`ORBextractor` keeps the reference's constructor arguments, call signature and getters
(/root/reference/code/include/ORBextractor.h:48-125): `extractor(image, mask) -> (keypoints, descriptors)`
with keypoints as a structured array laid out like cv::KeyPoint and descriptors as N x 32 uint8.
The C++ drop-in with the literal `operator()(cv::InputArray, ...)` signature lives in
swarmmap_b200/host/ORBextractor.h; this module is the same thin layer for Python callers, tests and bench.py.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import KP_DTYPE, SwmError, check, ptr

__all__ = ["ORBextractor", "KP_DTYPE", "SwmError"]


class ORBextractor:
    """ORB_SLAM2::ORBextractor(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST) on a B200."""

    HARRIS_SCORE, FAST_SCORE = 0, 1  # ORBextractor.h:52

    def __init__(self, nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST, device=0, max_batch=1,
                 max_fast_per_level=0, debug_score=False):
        self._lib = _lib.load()
        self.nfeatures, self.scaleFactor, self.nlevels = int(nfeatures), float(scaleFactor), int(nlevels)
        self.iniThFAST, self.minThFAST = int(iniThFAST), int(minThFAST)
        self.device, self.max_batch = int(device), int(max_batch)
        cfg = _lib.OrbCfg(self.nfeatures, self.scaleFactor, self.nlevels, self.iniThFAST, self.minThFAST,
                          self.max_batch, int(max_fast_per_level))
        h = C.c_void_p()
        rc = self._lib.swm_orb_create(C.byref(cfg), self.device, C.byref(h))
        check(rc, None, "swm_orb_create")
        self._h = h
        if debug_score:
            check(self._lib.swm_orb_set_debug(h, 1), h, "swm_orb_set_debug")
        n = self.nlevels
        self.mvScaleFactor = np.zeros(n, np.float32)
        self.mvInvScaleFactor = np.zeros(n, np.float32)
        self.mvLevelSigma2 = np.zeros(n, np.float32)
        self.mvInvLevelSigma2 = np.zeros(n, np.float32)
        check(self._lib.swm_orb_scale_tables(h, ptr(self.mvScaleFactor), ptr(self.mvInvScaleFactor),
                                              ptr(self.mvLevelSigma2), ptr(self.mvInvLevelSigma2)), h, "scale_tables")
        self.mnFeaturesPerLevel = np.zeros(n, np.int32)
        check(self._lib.swm_orb_level_quotas(h, ptr(self.mnFeaturesPerLevel)), h, "level_quotas")

    def close(self):
        if getattr(self, "_h", None):
            self._lib.swm_orb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- reference getters (ORBextractor.h:64-86)
    def GetLevels(self):
        return self.nlevels

    def GetScaleFactor(self):
        return self.scaleFactor

    def GetScaleFactors(self):
        return self.mvScaleFactor.copy()

    def GetInverseScaleFactors(self):
        return self.mvInvScaleFactor.copy()

    def GetScaleSigmaSquares(self):
        return self.mvLevelSigma2.copy()

    def GetInverseScaleSigmaSquares(self):
        return self.mvInvLevelSigma2.copy()

    def max_keypoints(self):
        return int(self._lib.swm_orb_max_keypoints(self._h))

    # ---- operator() (ORBextractor.cc:746-819); mask is ignored as in the reference
    def __call__(self, image, mask=None):
        if image is None or image.size == 0:
            return np.zeros(0, KP_DTYPE), np.zeros((0, 32), np.uint8)
        if image.dtype != np.uint8 or image.ndim != 2:
            raise TypeError("image must be CV_8UC1 (2-D uint8)")  # assert at ORBextractor.cc:754
        if image.strides[1] != 1:
            image = np.ascontiguousarray(image)
        hh, w = image.shape
        cap = self.max_keypoints()
        kps = np.empty(cap, KP_DTYPE)
        desc = np.empty((cap, 32), np.uint8)
        n = C.c_int(0)
        rc = self._lib.swm_orb_extract(self._h, ptr(image), w, hh, image.strides[0], ptr(kps), ptr(desc), cap,
                                       C.byref(n))
        check(rc, self._h, "swm_orb_extract")
        return kps[:n.value].copy(), desc[:n.value].copy()

    def extract_batch(self, images, out=None):
        """images: (B, H, W) uint8 host array.  Returns (kps (B,cap), desc (B,cap,32), n (B,))."""
        images = np.ascontiguousarray(images, np.uint8)
        b, hh, w = images.shape
        cap = self.max_keypoints() if out is None else out[0].shape[1]
        if out is None:
            kps = np.empty((b, cap), KP_DTYPE)
            desc = np.empty((b, cap, 32), np.uint8)
            n = np.zeros(b, np.int32)
        else:
            kps, desc, n = out
        rc = self._lib.swm_orb_extract_batch(self._h, ptr(images), b, w, hh, w, w * hh, ptr(kps), ptr(desc), cap,
                                             ptr(n))
        check(rc, self._h, "swm_orb_extract_batch")
        return kps, desc, n

    def extract_batch_async(self, images, out):
        """Enqueue one batch (<= max_batch frames, pinned host arrays) and return; call sync() before
        reading `out` = (kps (B,cap), desc (B,cap,32), n (B,))."""
        b, hh, w = images.shape
        kps, desc, n = out
        rc = self._lib.swm_orb_extract_batch_async(self._h, ptr(images), b, w, hh, images.strides[1],
                                                   images.strides[0], ptr(kps), ptr(desc), kps.shape[1], ptr(n))
        check(rc, self._h, "swm_orb_extract_batch_async")

    def sync(self):
        check(self._lib.swm_orb_sync(self._h), self._h, "swm_orb_sync")

    def extract_batch_device(self, d_imgs_ptr, batch, w, hh, stride, frame_stride, d_kps_ptr, d_desc_ptr, cap,
                             d_n_ptr, stream=None):
        rc = self._lib.swm_orb_extract_batch_device(self._h, d_imgs_ptr, batch, w, hh, stride, frame_stride,
                                                    d_kps_ptr, d_desc_ptr, cap, d_n_ptr, stream)
        check(rc, self._h, "swm_orb_extract_batch_device")

    def stereo_match(self, right, bf, b, batch):
        """Frame::ComputeStereoMatches (reference Frame.cc:516-690) for the batch this extractor (left view) and `right`
        (right view) extracted last: returns (mvuRight, mvDepth) as (batch, cap) float32 arrays, -1 = no match.
        `batch` must be the number of frames resident: extract_batch keeps only its last chunk of max_batch frames."""
        cap = self.max_keypoints()
        u = np.empty((batch, cap), np.float32)
        z = np.empty((batch, cap), np.float32)
        check(self._lib.swm_orb_stereo_match(self._h, right._h, bf, b, ptr(u), ptr(z), cap, batch), self._h,
              "swm_orb_stereo_match")
        return u, z

    def run_stage(self, mask, batch, stream=None):
        check(self._lib.swm_orb_run_stage(self._h, mask, batch, stream), self._h, "swm_orb_run_stage")

    def last_launches(self):
        return int(self._lib.swm_orb_last_launches(self._h))

    def level_ptr(self, frame, level, which):
        dev, w, hh, pitch = C.c_void_p(), C.c_int(), C.c_int(), C.c_int()
        check(self._lib.swm_orb_level_ptr(self._h, frame, level, which, C.byref(dev), C.byref(w), C.byref(hh),
                                          C.byref(pitch)), self._h, "swm_orb_level_ptr")
        return dev.value, w.value, hh.value, pitch.value

    # ---- parity introspection
    def debug_plane(self, frame, level, which):
        _, w, hh, _ = self.level_ptr(frame, level, 0)
        if which == 0:
            w, hh = w + 38, hh + 38
        out = np.empty((hh, w), np.uint8)
        check(self._lib.swm_orb_debug_plane(self._h, frame, level, which, ptr(out), w), self._h, "debug_plane")
        return out

    def debug_points(self, frame, level, which, cap=200000):
        buf = np.empty((cap, 3), np.int32)
        n = self._lib.swm_orb_debug_points(self._h, frame, level, which, ptr(buf), cap)
        if n < 0:
            check(n, self._h, "debug_points")
        return buf[:min(n, cap)].copy()
