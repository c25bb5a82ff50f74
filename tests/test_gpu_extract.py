"""GPU parity of the extractor against the CPU oracle, stage by stage (run with -m gpu on a B200).

Bar (BASELINE.json north_star): pyramid, FAST keypoint set, quadtree selection bit-exact;
orientation within 1e-4 rad; >= 99.9 % of descriptor bits identical.  On top of that bar every keypoint the GPU
returns is checked on its own against the float64 reference of tests/orb_ref.py (coordinates, size, response,
angle within 4e-6 rad, no descriptor bit that float32 rounding cannot explain).
"""
import numpy as np
import pytest

import orb_ref
from swarmmap_b200 import synth

pytestmark = pytest.mark.gpu

ANGLE_TOL_RAD = 1e-4
DESC_BIT_FRACTION = 0.999


def _extractors(oracle, nfeatures, max_batch=1, **kw):
    from swarmmap_b200.orb import ORBextractor
    gpu = ORBextractor(nfeatures, 1.2, 8, 20, 7, max_batch=max_batch, debug_score=True, **kw)
    cpu = oracle.Extractor(nfeatures, 1.2, 8, 20, 7)
    return gpu, cpu


def _check_frame(gpu, cpu, img, frame=0, kd=None):
    """Compares every intermediate of `frame` of the last GPU batch with the oracle run on img."""
    okps, odesc = cpu(img)
    for l in range(gpu.GetLevels()):
        np.testing.assert_array_equal(gpu.debug_plane(frame, l, 0), cpu.level(l, 0), err_msg=f"bordered plane L{l}")
        np.testing.assert_array_equal(gpu.debug_plane(frame, l, 2), cpu.level(l, 2), err_msg=f"FAST score map L{l}")
        np.testing.assert_array_equal(gpu.debug_plane(frame, l, 1), cpu.level(l, 1), err_msg=f"blurred plane L{l}")
        g = gpu.debug_points(frame, l, 0)
        o = cpu.level_fast(l)
        # raster order (y, then x); the reference keeps at most 10 000 per level (Fast.hpp:30)
        gset = sorted(map(tuple, g.tolist()), key=lambda t: (t[1], t[0]))[:10000]
        oset = sorted(zip(o["x"].tolist(), o["y"].tolist(), o["score"].tolist()), key=lambda t: (t[1], t[0]))
        assert gset == oset, f"FAST keypoint set differs at level {l}: {len(gset)} vs {len(oset)}"
        g = gpu.debug_points(frame, l, 1)
        o = cpu.level_selected(l)
        assert g.tolist() == [list(t) for t in zip(o["x"].tolist(), o["y"].tolist(), o["score"].tolist())], \
            f"quadtree selection (ordered) differs at level {l}"
    if kd is not None:
        kps, desc = kd
        assert len(kps) == len(okps)
        for fld in ("x", "y", "size", "response", "octave", "class_id"):
            np.testing.assert_array_equal(kps[fld], okps[fld], err_msg=fld)
        dang = np.abs(kps["angle"] - okps["angle"])
        dang = np.minimum(dang, 360.0 - dang)
        assert np.deg2rad(dang.max()) <= ANGLE_TOL_RAD, f"max angle error {dang.max()} deg"
        bits = np.unpackbits(desc ^ odesc).sum()
        frac = 1.0 - bits / float(desc.size * 8)
        assert frac >= DESC_BIT_FRACTION, f"descriptor bit agreement {frac}"
        st = orb_ref.check_extractor_frame(gpu, frame, kps, desc)
        print(f"float64 reference: {st['n']} keypoints, max angle error {st['max_angle_err_rad']:.2e} rad, "
              f"{st['ambiguous_bits']} ambiguous bits")
    return okps, odesc


def test_single_frame_config1(oracle, swm):
    gpu, cpu = _extractors(oracle, 1000)
    img = synth.make_frame(752, 480, 20220404)
    kps, desc = gpu(img)
    assert 900 <= len(kps) <= gpu.max_keypoints()
    _check_frame(gpu, cpu, img, 0, (kps, desc))
    # determinism: same frame again -> identical bytes
    kps2, desc2 = gpu(img)
    assert kps.tobytes() == kps2.tobytes() and desc.tobytes() == desc2.tobytes()


def test_single_frame_config2_kitti(oracle, swm):
    for nf in (2000, 4000):
        gpu, cpu = _extractors(oracle, nf)
        img = synth.make_frame(1241, 376, 20220405)
        kps, desc = gpu(img)
        _check_frame(gpu, cpu, img, 0, (kps, desc))


def test_product_config_without_debug_map(oracle, swm):
    """The shipped configuration keeps no score map and detects pass 1 at iniThFAST; same keypoints."""
    from swarmmap_b200.orb import ORBextractor
    rng = np.random.default_rng(3)
    low = (120 + 6 * rng.standard_normal((480, 752))).clip(0, 255).astype(np.uint8)
    low[100:300, 200:500] = synth.make_frame(752, 480, 5)[100:300, 200:500]
    for img, nf in ((synth.make_frame(752, 480, 20220404), 1000), (low, 1000), (synth.make_frame(1241, 376, 20220405), 2000)):
        gpu = ORBextractor(nf, 1.2, 8, 20, 7)
        cpu = oracle.Extractor(nf, 1.2, 8, 20, 7)
        kps, desc = gpu(img)
        okps, odesc = cpu(img)
        assert len(kps) == len(okps)
        for fld in ("x", "y", "size", "response", "octave"):
            np.testing.assert_array_equal(kps[fld], okps[fld])
        for l in range(8):
            g = sorted(map(tuple, gpu.debug_points(0, l, 0).tolist()))
            o = cpu.level_fast(l)
            assert g == sorted(zip(o["x"].tolist(), o["y"].tolist(), o["score"].tolist()))
        assert 1.0 - np.unpackbits(desc ^ odesc).sum() / float(desc.size * 8) >= DESC_BIT_FRACTION


def test_batch_matches_single(oracle, swm):
    gpu, cpu = _extractors(oracle, 1000, max_batch=4)
    imgs = synth.make_batch(6, 752, 480, 20220410)  # 6 frames through a batch-4 handle: two chunks
    kps, desc, n = gpu.extract_batch(imgs)
    for f in range(6):
        okps, odesc = cpu(imgs[f])
        assert n[f] == len(okps)
        for fld in ("x", "y", "size", "response", "octave"):
            np.testing.assert_array_equal(kps[f, :n[f]][fld], okps[fld])
        bits = np.unpackbits(desc[f, :n[f]] ^ odesc).sum()
        assert 1.0 - bits / float(odesc.size * 8) >= DESC_BIT_FRACTION
    # intermediates of the last chunk (frames 4,5 sit in slots 0,1)
    _check_frame(gpu, cpu, imgs[5], 1, (kps[5, :n[5]], desc[5, :n[5]]))


def test_bench_batch_size_invariances(oracle, swm):
    """Size-independent properties at the bench's handle batch (64 frames per call, the long-row-block / four-tile-run
    configuration of the kernels, which the small-batch tests above do not reach): a frame's result does not depend on
    its slot in the batch, on its neighbours, or on the run; a single-frame handle (8-row blocks, one tile per warp)
    gives the same bytes; and three sampled frames equal the oracle."""
    from swarmmap_b200.orb import ORBextractor
    base = synth.make_batch(16, 752, 480, 20220411)
    rng = np.random.default_rng(5)
    order = rng.integers(0, 16, 64)
    imgs = base[order]
    big = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=64)
    k1, d1, n1 = big.extract_batch(imgs)
    k2, d2, n2 = big.extract_batch(imgs[::-1].copy())  # same frames, reversed slots, second run
    one = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=1)
    first_slot = {}
    for s in range(64):
        f = int(order[s])
        r = 63 - s
        assert n1[s] == n2[r]
        assert k1[s, :n1[s]].tobytes() == k2[r, :n2[r]].tobytes() and d1[s, :n1[s]].tobytes() == d2[r, :n2[r]].tobytes()
        if f in first_slot:  # the same frame in another slot of the same batch
            t = first_slot[f]
            assert n1[s] == n1[t] and k1[s, :n1[s]].tobytes() == k1[t, :n1[t]].tobytes() and d1[s, :n1[s]].tobytes() == d1[t, :n1[t]].tobytes()
        else:
            first_slot[f] = s
    for f in (0, 7, 15):
        s = first_slot.get(f)
        if s is None:
            continue
        ks, ds = one(base[f])
        assert len(ks) == n1[s] and ks.tobytes() == k1[s, :n1[s]].tobytes() and ds.tobytes() == d1[s, :n1[s]].tobytes()
        okps, odesc = oracle.Extractor(1000, 1.2, 8, 20, 7)(base[f])
        assert len(okps) == n1[s]
        for fld in ("x", "y", "size", "response", "octave"):
            np.testing.assert_array_equal(k1[s, :n1[s]][fld], okps[fld])


# the layout limits of 8 levels at 1.2 (oracle.level_sizes): 200x138 has a 39 px coarsest level (the smallest side
# accepted); 528x140 gives DistributeOctTree round((W - 32) / (H - 32)) == 16 initial nodes on its coarsest level
# (the largest accepted; the live-node bound there is 4 x 16, not quota + 3); 4000 px is the widest level accepted
@pytest.mark.parametrize("w,h", [(640, 480), (333, 257), (200, 150), (1001, 301), (200, 138), (528, 140), (3990, 400),
                                 (4000, 400)])
def test_odd_sizes(oracle, swm, w, h):
    gpu, cpu = _extractors(oracle, 500)
    img = synth.make_frame(w, h, 1234 + w)
    kps, desc = gpu(img)
    _check_frame(gpu, cpu, img, 0, (kps, desc))


# one past each limit: a 38 px coarsest level, 17 initial quadtree nodes, a 4001 px level
@pytest.mark.parametrize("w,h", [(200, 137), (529, 140), (4001, 400)])
def test_sizes_past_the_limits_refused(swm, w, h):
    from swarmmap_b200.orb import ORBextractor, SwmError
    gpu = ORBextractor(500, 1.2, 8, 20, 7)
    with pytest.raises(SwmError, match="SWM_E_INVALID"):
        gpu(synth.make_frame(w, h, 1234 + w))
    kps, _ = gpu(synth.make_frame(640, 480, 1))  # the handle stays usable
    assert len(kps) > 400


def test_textureless_and_noise(oracle, swm):
    gpu, cpu = _extractors(oracle, 1000)
    flat = np.full((480, 752), 128, np.uint8)
    kps, desc = gpu(flat)
    assert len(kps) == 0 and desc.shape == (0, 32)
    # low-contrast frame: exercises the minThFAST tile retry everywhere
    rng = np.random.default_rng(3)
    low = (120 + 6 * rng.standard_normal((480, 752))).clip(0, 255).astype(np.uint8)
    low[100:300, 200:500] = synth.make_frame(752, 480, 5)[100:300, 200:500]
    kps, desc = gpu(low)
    _check_frame(gpu, cpu, low, 0, (kps, desc))
    # white noise: more FAST survivors than the reference's 10 000-entry buffer on level 0
    noise = rng.integers(0, 256, (480, 752), dtype=np.uint8)
    kps, desc = gpu(noise)
    _check_frame(gpu, cpu, noise, 0, (kps, desc))


def test_strided_input_and_empty(oracle, swm):
    gpu, cpu = _extractors(oracle, 1000)
    big = synth.make_frame(800, 500, 99)
    view = big[10:490, 20:772]  # non-contiguous rows (stride 800)
    kps, desc = gpu(view)
    okps, odesc = cpu(np.ascontiguousarray(view))
    np.testing.assert_array_equal(kps["x"], okps["x"])
    np.testing.assert_array_equal(kps["y"], okps["y"])
    k0, d0 = gpu(np.zeros((0, 0), np.uint8))
    assert len(k0) == 0
    with pytest.raises(TypeError):
        gpu(np.zeros((480, 752), np.float32))


def test_scale_tables_and_quotas(oracle, swm):
    gpu, cpu = _extractors(oracle, 1000)
    sf, inv, s2, inv2 = oracle.scale_tables(1.2, 8)
    np.testing.assert_array_equal(gpu.GetScaleFactors(), sf)
    np.testing.assert_array_equal(gpu.GetInverseScaleFactors(), inv)
    np.testing.assert_array_equal(gpu.GetScaleSigmaSquares(), s2)
    np.testing.assert_array_equal(gpu.GetInverseScaleSigmaSquares(), inv2)
    np.testing.assert_array_equal(gpu.mnFeaturesPerLevel, oracle.level_quotas(1000))
    assert gpu.GetLevels() == 8 and abs(gpu.GetScaleFactor() - 1.2) < 1e-6


@pytest.mark.parametrize("cfg", [(500, 1.3, 5, 15, 5), (1500, 1.1, 10, 30, 10), (300, 1.5, 3, 20, 7), (2000, 1.2, 8, 40, 20)])
def test_other_extractor_settings(oracle, swm, cfg):
    """Non-default ORBextractor.* settings (nFeatures, scaleFactor, nLevels, iniThFAST, minThFAST)."""
    from swarmmap_b200.orb import ORBextractor
    nf, sf, nl, ini, mn = cfg
    gpu = ORBextractor(nf, sf, nl, ini, mn, debug_score=True)
    cpu = oracle.Extractor(nf, sf, nl, ini, mn)
    img = synth.make_frame(640, 480, 77)
    kps, desc = gpu(img)
    okps, odesc = cpu(img)
    for l in range(nl):
        np.testing.assert_array_equal(gpu.debug_plane(0, l, 0), cpu.level(l, 0), err_msg=f"plane L{l}")
        np.testing.assert_array_equal(gpu.debug_plane(0, l, 1), cpu.level(l, 1), err_msg=f"blur L{l}")
        np.testing.assert_array_equal(gpu.debug_plane(0, l, 2), cpu.level(l, 2), err_msg=f"score L{l}")
    assert len(kps) == len(okps) and len(kps) > 100
    for fld in ("x", "y", "size", "response", "octave"):
        np.testing.assert_array_equal(kps[fld], okps[fld], err_msg=fld)
    assert 1.0 - np.unpackbits(desc ^ odesc).sum() / float(desc.size * 8) >= DESC_BIT_FRACTION
    np.testing.assert_array_equal(gpu.mnFeaturesPerLevel, oracle.level_quotas(nf, sf, nl))


# max per-level quota of nfeatures at 8 levels, 1.2 (oracle.level_quotas): 2359 -> 512, 2360 -> 513, 4717 -> 1024,
# 4718 -> 1025, 9432 -> 2048 (the largest accepted), i.e. both sides of each quadtree instantiation
# (ot_max_live(512 / 1024 / 2048)); one level of 2000 takes the 2048 instantiation with a single level
@pytest.mark.parametrize("cfg", [(2359, 1.2, 8, 20, 7), (2360, 1.2, 8, 20, 7), (4717, 1.2, 8, 20, 7),
                                 (4718, 1.2, 8, 20, 7), (9432, 1.2, 8, 20, 7), (2000, 1.2, 1, 20, 7)],
                         ids=["q512", "q513", "q1024", "q1025", "q2048", "q2000-1level"])
def test_quota_boundaries(oracle, swm, cfg):
    """White noise at 1241x376 leaves more level-0 FAST candidates than any quota, so the quadtree runs to the quota."""
    from swarmmap_b200.orb import ORBextractor
    nf, sf, nl, ini, mn = cfg
    q = oracle.level_quotas(nf, sf, nl)
    assert {2359: 512, 2360: 513, 4717: 1024, 4718: 1025, 9432: 2048, 2000: 2000}[nf] == q.max()
    gpu = ORBextractor(nf, sf, nl, ini, mn, debug_score=True)
    np.testing.assert_array_equal(gpu.mnFeaturesPerLevel, q)
    cpu = oracle.Extractor(nf, sf, nl, ini, mn)
    img = np.random.default_rng(nf).integers(0, 256, (376, 1241), dtype=np.uint8)
    kps, desc = gpu(img)
    _check_frame(gpu, cpu, img, 0, (kps, desc))
    assert (kps["octave"] == 0).sum() >= q[0]


def test_quota_past_2048_refused(oracle, swm):
    from swarmmap_b200.orb import ORBextractor, SwmError
    assert oracle.level_quotas(9433).max() == 2049
    with pytest.raises(SwmError, match="SWM_E_INVALID"):
        ORBextractor(9433, 1.2, 8, 20, 7)


def test_size_change_on_one_handle(oracle, swm):
    """The reference assumes one frame size per extractor (ORBextractor.h:89); the handle re-plans instead."""
    from swarmmap_b200.orb import ORBextractor
    gpu = ORBextractor(800, 1.2, 8, 20, 7)
    cpu = oracle.Extractor(800, 1.2, 8, 20, 7)
    for (w, h, seed) in ((752, 480, 1), (640, 360, 2), (752, 480, 3), (401, 299, 4)):
        img = synth.make_frame(w, h, seed)
        kps, desc = gpu(img)
        okps, odesc = cpu(img)
        assert len(kps) == len(okps)
        np.testing.assert_array_equal(kps["x"], okps["x"])
        np.testing.assert_array_equal(kps["response"], okps["response"])
        assert 1.0 - np.unpackbits(desc ^ odesc).sum() / float(desc.size * 8) >= DESC_BIT_FRACTION


def test_concurrent_handles_from_threads(oracle, swm):
    """One extractor per agent thread (swarm_map.cc:329-337): handles are independent and deterministic."""
    import threading
    from swarmmap_b200.orb import ORBextractor
    imgs = synth.make_batch(4, 752, 480, 123)
    cpu = oracle.Extractor(1000, 1.2, 8, 20, 7)
    ref = [cpu(im) for im in imgs]
    out = [None] * 4

    def agent(i):
        ex = ORBextractor(1000, 1.2, 8, 20, 7)
        res = None
        for _ in range(5):
            res = ex(imgs[i])
        out[i] = res

    ts = [threading.Thread(target=agent, args=(i,)) for i in range(4)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    for i in range(4):
        kps, desc = out[i]
        okps, odesc = ref[i]
        assert len(kps) == len(okps)
        for fld in ("x", "y", "response", "octave"):
            np.testing.assert_array_equal(kps[fld], okps[fld])
        assert 1.0 - np.unpackbits(desc ^ odesc).sum() / float(desc.size * 8) >= DESC_BIT_FRACTION


def test_small_caller_capacity(oracle, swm):
    """A caller buffer smaller than the keypoint count gets the first `cap` keypoints and n == cap."""
    import ctypes as C
    from swarmmap_b200.orb import ORBextractor
    from swarmmap_b200._lib import KP_DTYPE, ptr
    gpu = ORBextractor(1000, 1.2, 8, 20, 7)
    img = synth.make_frame(752, 480, 20220404)
    full_k, full_d = gpu(img)
    cap = 300
    kps = np.zeros(cap, KP_DTYPE)
    desc = np.zeros((cap, 32), np.uint8)
    n = C.c_int(0)
    rc = gpu._lib.swm_orb_extract(gpu._h, ptr(img), 752, 480, 752, ptr(kps), ptr(desc), cap, C.byref(n))
    assert rc == 0 and n.value == cap
    assert kps.tobytes() == full_k[:cap].tobytes() and (desc == full_d[:cap]).all()
