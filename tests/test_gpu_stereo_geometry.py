"""swm_orb_stereo_match at the launch geometries the benchmark uses, on every handle situation, and on hand-built
frames injected into the extractor's resident buffers.  Every frame is compared bit for bit with the second reading
(tests/stereo_ref.py) and, for extracted keypoints, with the oracle; the reading's trace is tallied over the file to
show which rules the device kernels were exercised on."""
import ctypes as C

import numpy as np
import pytest

from swarmmap_b200 import synth
import stereo_cases
import stereo_ref

pytestmark = pytest.mark.gpu

EUROC_BF, EUROC_FX = 47.90639384423901, 458.654
KITTI_BF, KITTI_FX = 386.1448, 718.856
TALLY = {k: 0 for k in stereo_ref.OUTCOMES + ("tie", "border")}
FRAMES = [0]


@pytest.fixture(scope="module")
def tables(oracle):
    sf, inv_sf, _, _ = oracle.scale_tables(1.2, 8)
    return sf, inv_sf


def _planes(ex, f):
    """mvImagePyramid[l] of frame f after operator(): the bordered un-blurred buffer with the level blurred in place."""
    out = []
    for l in range(ex.nlevels):
        buf = ex.debug_plane(f, l, 0).copy()
        buf[19:-19, 19:-19] = ex.debug_plane(f, l, 1)
        out.append(buf)
    return out


def _check(oracle, tables, exl, exr, frames, u, z, mbf, mb, with_oracle=True):
    """frames: per frame (kl, dl, kr, dr) as the kernel read them.  Returns the reading's u per frame."""
    sf, inv_sf = tables
    out = []
    for f, (kl, dl, kr, dr) in enumerate(frames):
        pl, pr = _planes(exl, f), _planes(exr, f)
        u1, z1, n1, tr = stereo_ref.stereo_matches(kl, dl, kr, dr, pl, pr, sf, inv_sf, mbf, mb)
        n = len(kl)
        np.testing.assert_array_equal(u[f, :n].view(np.uint32), u1.view(np.uint32), err_msg=f"mvuRight frame {f}")
        np.testing.assert_array_equal(z[f, :n].view(np.uint32), z1.view(np.uint32), err_msg=f"mvDepth frame {f}")
        if with_oracle:
            u0, z0, n0 = oracle.stereo_matches(kl, dl, kr, dr, pl, pr, sf, inv_sf, mbf, mb)
            assert np.array_equal(u0.view(np.uint32), u1.view(np.uint32)) and n0 == n1, f"oracle frame {f}"
        stereo_ref.tally(tr, TALLY)
        FRAMES[0] += 1
        out.append(u1)
    return out


def _extracted(kl, dl, nl, kr, dr, nr):
    return [(kl[f, :nl[f]], dl[f, :nl[f]], kr[f, :nr[f]], dr[f, :nr[f]]) for f in range(len(nl))]


def _run_batch(oracle, tables, lefts, rights, nfeat, mbf, fx, max_batch=None, nfeat_r=None, max_batch_r=None):
    from swarmmap_b200.orb import ORBextractor
    B = len(lefts)
    exl = ORBextractor(nfeat, 1.2, 8, 20, 7, max_batch=max_batch or B)
    exr = ORBextractor(nfeat_r or nfeat, 1.2, 8, 20, 7, max_batch=max_batch_r or max_batch or B)
    kl, dl, nl = exl.extract_batch(np.stack(lefts))
    kr, dr, nr = exr.extract_batch(np.stack(rights))
    u, z = exl.stereo_match(exr, mbf, mbf / fx, B)
    ref = _check(oracle, tables, exl, exr, _extracted(kl, dl, nl, kr, dr, nr), u, z, mbf, mbf / fx)
    return u, z, nl, ref


def test_benchmark_geometry_32_different_pairs(oracle, tables):
    """One call of 32 different pairs at 752 x 480, 1000 features, max_batch 32; slot 31 repeats slot 0."""
    kinds = [{}, {"d_near": 9.0, "d_far": 0.0}, {"right_shift": 6}, {"d_near": 30.0, "d_far": 20.0},
             {"d_near": 60.0, "d_far": 10.0}, {"d_near": 3.0, "d_far": 0.0, "right_shift": 1}]
    lefts, rights = [], []
    for s in range(31):
        l, r = synth.make_stereo_pair(752, 480, 500 + s, **kinds[s % len(kinds)])
        lefts.append(l)
        rights.append(r)
    lefts.append(lefts[0])
    rights.append(rights[0])
    u, z, nl, _ = _run_batch(oracle, tables, lefts, rights, 1000, EUROC_BF, EUROC_FX)
    assert np.array_equal(u[0, :nl[0]].view(np.uint32), u[31, :nl[31]].view(np.uint32))
    assert np.array_equal(z[0, :nl[0]].view(np.uint32), z[31, :nl[31]].view(np.uint32))
    assert sum((u[f, :nl[f]] >= 0).sum() for f in range(32)) > 100 * 16


def test_benchmark_input_every_row(oracle, tables):
    """bench.py's own stereo input (32 copies of one pair): all 32 rows, not only row 0, equal the reading."""
    l, r = synth.make_stereo_pair(752, 480, 20220421)
    u, z, nl, ref = _run_batch(oracle, tables, [l] * 32, [r] * 32, 1000, EUROC_BF, EUROC_FX)
    for f in range(32):
        assert np.array_equal(u[f, :nl[f]].view(np.uint32), ref[0].view(np.uint32)), f


def test_kitti_geometry_and_wide_band(oracle, tables):
    lefts, rights = zip(*[synth.make_stereo_pair(1241, 376, 40 + s, d_near=70.0, d_far=2.0 + s) for s in range(8)])
    _run_batch(oracle, tables, list(lefts), list(rights), 2000, KITTI_BF, KITTI_FX)
    # maxD = 47.9 / (47.9 / 2000) = 2000 px > width: every right keypoint of the row band is a candidate
    lefts, rights = zip(*[synth.make_stereo_pair(752, 480, 60 + s, d_near=30.0, d_far=25.0) for s in range(4)])
    _run_batch(oracle, tables, list(lefts), list(rights), 800, 47.9, 2000.0)


@pytest.mark.parametrize("nfeat_l,nfeat_r,mb_l,mb_r", [(1000, 2000, 3, 2), (2000, 1000, 2, 3)])
def test_handles_with_different_capacities(oracle, tables, nfeat_l, nfeat_r, mb_l, mb_r):
    lefts, rights = zip(*[synth.make_stereo_pair(752, 480, 80 + s) for s in range(2)])
    _run_batch(oracle, tables, list(lefts), list(rights), nfeat_l, EUROC_BF, EUROC_FX, max_batch=mb_l, nfeat_r=nfeat_r,
               max_batch_r=mb_r)


def test_single_frame_operator_run_capture_replay(oracle, tables):
    """The C++ drop-in's path: operator() per view, then stereo_match(..., 1).  The first call runs the launches,
    the second captures them into a CUDA graph, the third replays it."""
    from swarmmap_b200.orb import ORBextractor
    exl = ORBextractor(1000, 1.2, 8, 20, 7)
    exr = ORBextractor(1000, 1.2, 8, 20, 7)
    for s in range(3):
        l, r = synth.make_stereo_pair(752, 480, 90 + s, d_near=20.0 + 5 * s)
        kl, dl = exl(l)
        kr, dr = exr(r)
        u, z = exl.stereo_match(exr, EUROC_BF, EUROC_BF / EUROC_FX, 1)
        ref = _check(oracle, tables, exl, exr, [(kl, dl, kr, dr)], u, z, EUROC_BF, EUROC_BF / EUROC_FX)
        assert (ref[0] >= 0).sum() > 100


def _device_buffers(torch, B, cap):
    return (torch.empty((B, cap, 28), dtype=torch.uint8, device="cuda"),
            torch.empty((B, cap, 32), dtype=torch.uint8, device="cuda"),
            torch.empty(B, dtype=torch.int32, device="cuda"))


def _extract_device(ex, torch, imgs, bufs, stream=None):
    d_imgs = torch.from_numpy(np.ascontiguousarray(imgs)).cuda()
    torch.cuda.synchronize()  # the upload is on torch's stream, the extraction on another
    B, H, W = imgs.shape
    k, d, n = bufs
    ex.extract_batch_device(d_imgs.data_ptr(), B, W, H, W, W * H, k.data_ptr(), d.data_ptr(), k.shape[1], n.data_ptr(),
                            stream)
    return d_imgs


def _download(bufs):
    from swarmmap_b200._lib import KP_DTYPE
    k, d, n = (t.cpu().numpy() for t in bufs)
    return np.ascontiguousarray(k).view(KP_DTYPE)[..., 0], d, n


def test_right_view_in_flight_on_side_stream(oracle, tables):
    """The right view is extracted on a side stream and stereo_match is called without synchronising: the left
    handle's stream waits for it on an event."""
    import torch
    from swarmmap_b200.orb import ORBextractor
    B = 4
    lefts, rights = zip(*[synth.make_stereo_pair(752, 480, 100 + s) for s in range(B)])
    exl = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=B)
    exr = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=B)
    exl.extract_batch(np.stack(lefts))  # sizes the handles: max_keypoints() is a looser bound before the first frame
    exr.extract_batch(np.stack(rights))
    cap = exl.max_keypoints()
    bl, br = _device_buffers(torch, B, cap), _device_buffers(torch, B, cap)
    side = torch.cuda.Stream()
    keep = _extract_device(exl, torch, np.stack(lefts), bl)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        keep_r = _extract_device(exr, torch, np.stack(rights), br, C.c_void_p(side.cuda_stream))
    u, z = exl.stereo_match(exr, EUROC_BF, EUROC_BF / EUROC_FX, B)
    torch.cuda.synchronize()
    del keep, keep_r
    kl, dl, nl = _download(bl)
    kr, dr, nr = _download(br)
    _check(oracle, tables, exl, exr, _extracted(kl, dl, nl, kr, dr, nr), u, z, EUROC_BF, EUROC_BF / EUROC_FX)


# ---- hand-built frames injected into the resident buffers

def _assert_injectable(kps, n, ex, cap):
    """Every injected keypoint keeps each window read of the kernel inside the 19-px border of its plane."""
    inv = ex.mvInvScaleFactor
    for f in range(len(n)):
        assert 0 <= n[f] <= cap
        k = kps[f, :n[f]]
        assert ((k["octave"] >= 0) & (k["octave"] < ex.nlevels)).all()
        for lev in np.unique(k["octave"]):
            _, w, h, _ = ex.level_ptr(f, int(lev), 0)
            s = k[k["octave"] == lev]
            x = stereo_ref.c_round(s["x"] * inv[lev])
            y = stereo_ref.c_round(s["y"] * inv[lev])
            assert ((x >= 0) & (x <= w - 1) & (y >= 0) & (y <= h - 1)).all(), (f, lev)


def _full_frame(cap, sf, seed):
    """cap left and cap right keypoints on a shifted pair: most of them match."""
    rng = np.random.default_rng(seed)
    kl = np.zeros(cap, stereo_cases.KP_DTYPE)
    kr = np.zeros(cap, stereo_cases.KP_DTYPE)
    kl["x"] = rng.integers(30, stereo_cases.W - 30, cap).astype(np.float32)
    kl["y"] = rng.integers(20, stereo_cases.H - 20, cap).astype(np.float32)
    kr["x"] = kl["x"] - np.float32(2) - rng.integers(0, 3, cap).astype(np.float32)
    kr["y"] = kl["y"]
    kl["octave"] = kr["octave"] = 0
    kl["class_id"] = kr["class_id"] = -1
    dl = rng.integers(0, 256, (cap, 32), dtype=np.uint8)
    dr = dl.copy()
    dr[:, :2] ^= rng.integers(0, 256, (cap, 2), dtype=np.uint8)
    return kl, dl, kr, dr


def test_hand_built_cases_on_device(oracle, tables):
    import torch
    from swarmmap_b200._lib import KP_DTYPE
    from swarmmap_b200.orb import ORBextractor
    sf, inv_sf = tables
    cases = stereo_cases.build_cases(sf)
    pairs = [stereo_cases.make_pair(**c.pair) for c in cases]
    pairs += [stereo_cases.make_pair(D=4, seed=30)] * 3          # n_l = 0, n_r = 0, filled to cap
    B, CAP = len(pairs), 256
    exl = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=B)
    exr = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=B)
    bl, br = _device_buffers(torch, B, CAP), _device_buffers(torch, B, CAP)
    imgs = [_extract_device(exl, torch, np.stack([p[0] for p in pairs]), bl),
            _extract_device(exr, torch, np.stack([p[1] for p in pairs]), br)]
    torch.cuda.synchronize()
    planes = [(_planes(exl, f), _planes(exr, f)) for f in range(B)]
    frames = []
    for f, c in enumerate(cases):
        if c.needs_planes:
            c.needs_planes(c, *planes[f], sf, inv_sf)
        frames.append(c.arrays())
    kl, dl, kr, dr = frames[0]
    frames.append((kl[:0], dl[:0], kr, dr))
    frames.append((kl, dl, kr[:0], dr[:0]))
    frames.append(_full_frame(CAP, sf, 7))
    host = []
    for side in (0, 2):
        k = np.zeros((B, CAP), KP_DTYPE)
        d = np.zeros((B, CAP, 32), np.uint8)
        n = np.zeros(B, np.int32)
        for f, fr in enumerate(frames):
            n[f] = len(fr[side])
            k[f, :n[f]] = fr[side]
            d[f, :n[f]] = fr[side + 1]
        host.append((k, d, n))
    assert host[0][2][-1] == CAP and host[1][2][-1] == CAP
    _assert_injectable(host[0][0], host[0][2], exl, CAP)
    _assert_injectable(host[1][0], host[1][2], exr, CAP)
    torch.cuda.synchronize()
    for (k, d, n), bufs in zip(host, (bl, br)):
        bufs[0].copy_(torch.from_numpy(k.view(np.uint8).reshape(B, CAP, 28)))
        bufs[1].copy_(torch.from_numpy(d))
        bufs[2].copy_(torch.from_numpy(n))
    torch.cuda.synchronize()
    injected = _extracted(host[0][0], host[0][1], host[0][2], host[1][0], host[1][1], host[1][2])
    for call, (mbf, mb) in enumerate(stereo_cases.CALLS):
        u, z = exl.stereo_match(exr, mbf, mb, B)
        _check(oracle, tables, exl, exr, injected, u, z, mbf, mb)
        for f, c in enumerate(cases):  # the device result shows the intended outcome of each case
            for i, e in c.expect[call].items():
                got = u[f, i] >= 0
                assert got == (e in ("kept", "clamped")), (c.name, call, i, e)
    del imgs


# ---- the row contract of swm_orb_stereo_match

def test_stereo_match_refuses_other_row_counts(swm):
    from swarmmap_b200._lib import SwmError
    from swarmmap_b200.orb import ORBextractor
    lefts, rights = zip(*[synth.make_stereo_pair(752, 480, 120 + s) for s in range(5)])
    exl = ORBextractor(500, 1.2, 8, 20, 7, max_batch=3)
    exr = ORBextractor(500, 1.2, 8, 20, 7, max_batch=3)
    exl.extract_batch(np.stack(lefts[:3]))
    exr.extract_batch(np.stack(rights[:3]))
    with pytest.raises(SwmError, match="SWM_E_CAPACITY"):
        exl.stereo_match(exr, EUROC_BF, EUROC_BF / EUROC_FX, 1)
    u, _ = exl.stereo_match(exr, EUROC_BF, EUROC_BF / EUROC_FX, 3)
    assert u.shape[0] == 3
    for bf, b in ((0.0, 0.1), (-1.0, 0.1), (EUROC_BF, float("nan"))):
        with pytest.raises(SwmError, match="SWM_E_INVALID"):
            exl.stereo_match(exr, bf, b, 3)
    # 5 frames through max_batch = 2: only the last chunk (1 frame) stays resident
    a = ORBextractor(500, 1.2, 8, 20, 7, max_batch=2)
    b = ORBextractor(500, 1.2, 8, 20, 7, max_batch=2)
    a.extract_batch(np.stack(lefts))
    b.extract_batch(np.stack(rights))
    with pytest.raises(SwmError, match="extracted batch of 1 frames"):
        a.stereo_match(b, EUROC_BF, EUROC_BF / EUROC_FX, 5)


def test_stereo_match_refuses_65536_keypoint_rows(swm):
    import torch
    from swarmmap_b200._lib import SwmError
    from swarmmap_b200.orb import ORBextractor
    l, r = synth.make_stereo_pair(752, 480, 130)
    exl = ORBextractor(500, 1.2, 8, 20, 7)
    exr = ORBextractor(500, 1.2, 8, 20, 7)
    bl, br = _device_buffers(torch, 1, 65536), _device_buffers(torch, 1, 65536)
    keep = [_extract_device(exl, torch, l[None], bl), _extract_device(exr, torch, r[None], br)]
    torch.cuda.synchronize()
    with pytest.raises(SwmError, match="more than 65535"):
        exl.stereo_match(exr, EUROC_BF, EUROC_BF / EUROC_FX, 1)
    del keep


def test_zz_every_rule_reached_on_the_device():
    """Tallies of the reading's trace over every frame of this file that the device kernels computed."""
    if FRAMES[0] == 0:
        pytest.skip("no frame of this file ran")
    print(f"\nstereo trace over {FRAMES[0]} device frames: {TALLY}")
    missing = [k for k, v in TALLY.items() if v == 0 and k != "delta"]  # |deltaR| > 1 cannot fire (stereo_ref)
    assert not missing, (missing, TALLY)
    assert TALLY["delta"] == 0
