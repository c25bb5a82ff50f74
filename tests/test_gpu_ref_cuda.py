"""Pins the oracle's FAST / IC_Angle / rBRIEF restatements to the REFERENCE'S OWN CUDA kernels: code/src/cuda/Fast_gpu.cu
and Orb_gpu.cu compiled UNMODIFIED by nvcc for sm_100a with the reference's -use_fast_math (oracle/ref_cuda_wrap.cu ->
oracle/_ref/libref_cuda.so, built by `make -C oracle ref` where /root/reference exists; the .so travels to the GPU box).

What is compared, and how the reference kernel's races (SURVEY.md F5) are kept out of it:
  * per-pixel corner test + score (isKeyPoint2 / cornerScore, Fast_gpu.cu:190-262): a kernel of the wrapper calls the
    reference's device function on every pixel -- deterministic, full frames, bit-exact against orc_fast_score_map;
  * tile retry + NMS + emit (tileCalcKeypoints_kernel :284-341): on SINGLE-TILE images (38 x 38: one 32 x 32 block) the
    kernel has no inter-block race and its only nondeterminism is the atomicInc output order, so the sorted keypoint
    set must equal orc_fast_tile_select's exactly (incl. tiles that retry at minThFAST);
  * on whole level ROIs the kernel does race across tile borders (a block may read a neighbour's score before it is
    written or after the neighbour's retry pass rewrote it).  The oracle's lock-step definition is what the kernel
    produces when no such read is early or late; it is checked EXACTLY by running the kernel's four phases as four
    launches built from the reference's own device functions (isKeyPoint2, isMax; oracle/ref_cuda_wrap.cu
    refc_fast_detect_lockstep): keypoint set and per-tile retry flags identical on whole ROIs.  The original racy
    launch is run too and reported (measured on a B200: 43 of ~1970 keypoints in 20 of 322 tiles at level 0), with a
    loose bound;
  * IC_Angle_kernel + addBorder_kernel (:403-471): pt / octave / size bit-exact, angle within 1e-4 rad;
  * calcOrb_kernel (Orb_gpu.cu:67-100): >= 99.9 % of descriptor bits (its cosf / sinf are the fast-math intrinsics).
"""
import ctypes as C
import os

import numpy as np
import pytest

from swarmmap_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libref_cuda.so")
XLIB = os.path.join(ROOT, "oracle", "_ref", "liborbextractor_ref.so")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def refc():
    if not os.path.exists(LIB):
        pytest.skip("needs oracle/_ref/libref_cuda.so, compiled by `make -C oracle ref` "
                    "from the reference project's sources, which the repository does not contain")
    L = C.CDLL(LIB)
    assert L.refc_device_ok()
    L.refc_fast_score_map.restype = None
    L.refc_ic_angle.restype = None
    L.refc_orb.restype = None
    return L


@pytest.fixture(scope="module")
def ref_tables():
    """umax and the rBRIEF pattern as the reference's own ORBextractor constructor hands them to the GPU."""
    if not os.path.exists(XLIB):
        pytest.skip("needs oracle/_ref/liborbextractor_ref.so, compiled by `make -C oracle ref` "
                    "from the reference project's sources, which the repository does not contain")
    X = C.CDLL(XLIB)
    X.ref_orb_create.restype = C.c_void_p
    X.ref_orb_create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
    X.ref_orb_destroy.argtypes = [C.c_void_p]
    X.ref_orb_tables.argtypes = [C.c_void_p] * 8
    e = X.ref_orb_create(1000, 1.2, 8, 20, 7)
    t = [np.zeros(8, np.float32) for _ in range(4)]
    q = np.zeros(8, np.int32)
    um = np.zeros(16, np.int32)
    pat = np.zeros(1024, np.int8)
    X.ref_orb_tables(e, _p(t[0]), _p(t[1]), _p(t[2]), _p(t[3]), _p(q), _p(um), _p(pat))
    X.ref_orb_destroy(e)
    return um, np.ascontiguousarray(pat.astype(np.int32))  # 512 cv::Point (int x, y)


@pytest.fixture(scope="module")
def extracted(oracle):
    img = synth.make_frame(752, 480, 20220404)
    cpu = oracle.Extractor(1000, 1.2, 8, 20, 7)
    kps, desc = cpu(img)
    return cpu, kps, desc


def fast_detect(refc, img, hi=20, lo=7, cap=10000):
    img = np.ascontiguousarray(img)
    out = np.zeros((cap, 3), np.int32)
    n = refc.refc_fast_detect(_p(img), img.shape[1], img.shape[0], img.strides[0], hi, lo, cap, _p(out), cap)
    pts = out[:min(n, cap)]
    return n, sorted(map(tuple, pts.tolist()), key=lambda t: (t[1], t[0]))


@pytest.mark.parametrize("level", [0, 3, 7])
def test_score_map_equals_reference_device_code(oracle, refc, extracted, level):
    cpu = extracted[0]
    plane = cpu.level(level, 0)
    img = np.ascontiguousarray(plane[19:-19, 19:-19])
    h, w = img.shape
    for th in (7, 20):
        got = np.zeros((h, w), np.int32)
        refc.refc_fast_score_map(_p(img), w, h, img.strides[0], th, _p(got))
        exp = oracle.fast_score_map(img, 7).astype(np.int32)
        if th == 20:
            exp = np.where(exp >= 20, exp, 0)
        assert (exp > 0).sum() > 50
        np.testing.assert_array_equal(got, exp)


def test_single_tile_keypoint_sets_equal_reference_kernel(oracle, refc, extracted):
    """38 x 38 crops = exactly one block of tileCalcKeypoints_kernel: race-free, so the sets must be identical."""
    cpu = extracted[0]
    rng = np.random.default_rng(7)
    retried = with_kp = 0
    for trial in range(250):
        level = int(rng.integers(0, 8))
        plane = cpu.level(level, 0)
        H, W = plane.shape
        y0, x0 = int(rng.integers(0, H - 38)), int(rng.integers(0, W - 38))
        crop = np.ascontiguousarray(plane[y0:y0 + 38, x0:x0 + 38])
        if trial % 5 == 4:  # flatten the contrast so that nothing reaches iniThFAST and the tile retries
            crop = np.ascontiguousarray((crop.astype(np.int32) - 128) // 3 + 128).astype(np.uint8)
        n, got = fast_detect(refc, crop)
        score = oracle.fast_score_map(crop, 7)
        exp, retry = oracle.fast_tile_select(score, 20, want_retry=True)
        exp = sorted(zip(exp["x"].tolist(), exp["y"].tolist(), exp["score"].tolist()), key=lambda t: (t[1], t[0]))
        assert got == exp, (trial, level, y0, x0)
        retried += int(retry.any())
        with_kp += int(len(exp) > 0)
    assert retried > 20 and with_kp > 150, (retried, with_kp)


@pytest.mark.parametrize("level", [0, 1, 2, 4, 7])
def test_whole_roi_lockstep_of_reference_device_code(oracle, refc, extracted, level):
    cpu = extracted[0]
    plane = cpu.level(level, 0)
    roi = np.ascontiguousarray(plane[19 + 16:-(19 + 16), 19 + 16:-(19 + 16)])  # [16, w-16) x [16, h-16)
    h, w = roi.shape
    tiles_x, tiles_y = (w - 6 + 31) // 32, (h - 6 + 31) // 32
    out = np.zeros((10000, 3), np.int32)
    has_kp = np.zeros((tiles_y, tiles_x), np.uint8)
    n = refc.refc_fast_detect_lockstep(_p(roi), w, h, roi.strides[0], 20, 7, _p(out), 10000, _p(has_kp))
    got = sorted(map(tuple, out[:n].tolist()), key=lambda t: (t[1], t[0]))
    o = cpu.level_fast(level)
    exp = sorted(zip(o["x"].tolist(), o["y"].tolist(), o["score"].tolist()), key=lambda t: (t[1], t[0]))
    assert len(exp) > 50 and got == exp
    score = oracle.fast_score_map(roi, 7)
    _, retry = oracle.fast_tile_select(score, 20, want_retry=True)
    np.testing.assert_array_equal(has_kp == 0, retry[:tiles_y, :tiles_x] != 0)


@pytest.mark.parametrize("level", [0, 2, 5])
def test_whole_roi_racy_launch_is_close_to_lockstep(oracle, refc, extracted, level):
    cpu = extracted[0]
    plane = cpu.level(level, 0)
    roi = np.ascontiguousarray(plane[19 + 16:-(19 + 16), 19 + 16:-(19 + 16)])  # [16, w-16) x [16, h-16)
    n, got = fast_detect(refc, roi)
    o = cpu.level_fast(level)
    exp = set(zip(o["x"].tolist(), o["y"].tolist(), o["score"].tolist()))
    diff = set(got) ^ exp
    tiles = {((x - 3) // 32, (y - 3) // 32) for x, y, _ in diff}
    n_tiles = ((roi.shape[1] - 6 + 31) // 32) * ((roi.shape[0] - 6 + 31) // 32)
    print(f"level {level}: reference kernel {len(got)} keypoints, lock-step oracle {len(exp)}, "
          f"{len(diff)} differ in {len(tiles)} of {n_tiles} tiles")
    assert len(exp) > 100
    assert len(tiles) <= max(2, int(0.15 * n_tiles)), (len(tiles), n_tiles)


def test_ic_angle_equals_reference_kernel(oracle, refc, ref_tables, extracted):
    cpu = extracted[0]
    umax = ref_tables[0]
    sf = oracle.scale_tables(1.2, 8)[0]
    total = 0
    worst = 0.0
    for level in range(8):
        plane = cpu.level(level, 0)
        img = np.ascontiguousarray(plane[19:-19, 19:-19])
        sel = cpu.level_selected(level)
        n = len(sel["x"])
        kps = np.zeros(n, dtype=[("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                                 ("octave", "<i4"), ("class_id", "<i4")])
        kps["x"], kps["y"], kps["response"] = sel["x"], sel["y"], sel["score"]
        kps["size"], kps["angle"], kps["class_id"] = 7.0, -1.0, -1
        size = int(np.float32(31.0) * sf[level])  # ORBextractor.cc:717, int parameter
        refc.refc_ic_angle(_p(img), img.shape[1], img.shape[0], img.strides[0], _p(kps), n, 15, 16, 16, level, size,
                           _p(umax), 16)
        np.testing.assert_array_equal(kps["x"], sel["x"].astype(np.float32) + 16)
        np.testing.assert_array_equal(kps["y"], sel["y"].astype(np.float32) + 16)
        assert (kps["octave"] == level).all() and (kps["size"] == np.float32(size)).all()
        for i in range(n):
            a = oracle.ic_angle(img, int(kps["x"][i]), int(kps["y"][i]))
            d = abs(float(kps["angle"][i]) - a)
            worst = max(worst, min(d, 360.0 - d))
        total += n
    print(f"IC_Angle_kernel vs oracle: {total} keypoints, max difference {worst:.3e} deg")
    assert total > 900 and np.deg2rad(worst) <= 1e-4


def test_rbrief_equals_reference_kernel(oracle, refc, ref_tables, extracted):
    cpu, okps, odesc = extracted
    pattern = ref_tables[1]
    bits = total = 0
    for level in range(8):
        plane = cpu.level(level, 0).copy()           # bordered, un-blurred
        plane[19:-19, 19:-19] = cpu.level(level, 1)  # the blur is applied in place on the ROI only (ORBextractor.cc:719)
        plane = np.ascontiguousarray(plane)
        m = okps["octave"] == level
        n = int(m.sum())
        if n == 0:
            continue
        sf = oracle.scale_tables(1.2, 8)[0][level]
        kps = np.zeros(n, dtype=[("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                                 ("octave", "<i4"), ("class_id", "<i4")])
        # level coordinates of the selected keypoints (the extractor scales pt only after describing, :808-814)
        sel = cpu.level_selected(level)
        assert len(sel["x"]) == n
        kps["x"] = sel["x"].astype(np.float32) + 16 + 19  # + border of the uploaded plane
        kps["y"] = sel["y"].astype(np.float32) + 16 + 19
        kps["angle"] = okps["angle"][m]
        desc = np.zeros((n, 32), np.uint8)
        refc.refc_orb(_p(plane), plane.shape[1], plane.shape[0], plane.strides[0], _p(kps), n, _p(pattern), _p(desc))
        bits += int(np.unpackbits(desc ^ odesc[m]).sum())
        total += n * 256
    frac = 1.0 - bits / total
    print(f"calcOrb_kernel (-use_fast_math) vs oracle: {total // 256} descriptors, bit agreement {frac:.6f}")
    assert total > 900 * 256 and frac >= 0.999
