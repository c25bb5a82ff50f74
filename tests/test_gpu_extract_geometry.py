"""The extractor at the launch geometries the benchmark runs (run with -m gpu on a B200).

Launch geometry depends on the handle and on the call: the pyramid walk's row blocks on the call's batch and the SM
count, FAST's tiles per warp on the handle's max_batch (4 from 8 frames up, 1 below), the persistent FAST pass-2
grid on the batch, and pass 1's kernel on whether the handle keeps a score map.  Whatever the geometry, a frame's
keypoints and descriptors must be the bytes a single-frame handle gives (1 tile per warp, 8-row blocks, graph
replay), every keypoint must pass the float64 reference of tests/orb_ref.py, and sampled frames must equal the CPU
oracle stage by stage.
"""
import numpy as np
import pytest

import orb_ref
from swarmmap_b200 import synth
from test_gpu_extract import _check_frame

pytestmark = pytest.mark.gpu

W, H = 752, 480
SLOT_LOW, SLOT_NOISE, SLOT_FLAT, SLOT_SWEEP = 37, 101, 150, 200


def low_and_noise(w=W, h=H):
    """The low-contrast frame (minThFAST retry in almost every tile) and the white-noise frame (more FAST survivors
    than the reference's 10 000-entry buffer) of test_gpu_extract.test_textureless_and_noise, at any size."""
    rng = np.random.default_rng(3)
    low = (120 + 6 * rng.standard_normal((h, w))).clip(0, 255).astype(np.uint8)
    low[100:300, 200:500] = synth.make_frame(w, h, 5)[100:300, 200:500]
    noise = rng.integers(0, 256, (h, w), dtype=np.uint8)
    return low, noise


def angle_sweep_frame(w=W, h=H, cell=32, radius=9.0):
    """A grid of 32x32 patches, each holding a bright half-disc rotated to its own angle (evenly spread over
    [0, 360), with the multiples of 45 degrees exact), rendered with 4x4 supersampling so that rotations by less than
    a pixel still change the patch."""
    nx, ny = w // cell, h // cell
    n = nx * ny
    ang = np.arange(n) * (360.0 / n)
    for k in range(8):
        ang[int(np.argmin(np.abs(ang - 45.0 * k)))] = 45.0 * k
    ss = 4
    yy, xx = (np.mgrid[0:cell * ss, 0:cell * ss] + 0.5) / ss - cell / 2.0
    img = np.full((h, w), 96.0)
    for i in range(n):
        t = np.deg2rad(ang[i])
        u = xx * np.cos(t) + yy * np.sin(t)
        v = -xx * np.sin(t) + yy * np.cos(t)
        blob = ((u * u + v * v <= radius * radius) & (u >= 0)).astype(np.float64)
        cy, cx = divmod(i, nx)
        img[cy * cell:(cy + 1) * cell, cx * cell:(cx + 1) * cell] = 96.0 + 120.0 * blob.reshape(cell, ss, cell, ss).mean((1, 3))
    return np.rint(img).astype(np.uint8)


def _rows(kps, desc, n, s):
    return kps[s, :n[s]], desc[s, :n[s]]


def _same(a, b):
    return len(a[0]) == len(b[0]) and a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes()


def _report(total, what):
    print(f"{what}: float64 reference on {total['n']} keypoints, max angle error {total['max_angle_err_rad']:.2e} rad, "
          f"{total['ambiguous_bits']} ambiguous bits")


@pytest.fixture(scope="module")
def headline(swm):
    """256 frames of 752x480 as one call of the benchmark's headline handle would see them, with the hard inputs in
    some slots, and each frame's result from a single-frame handle."""
    from swarmmap_b200.orb import ORBextractor
    frames = synth.make_batch(256, W, H, 20220412)
    frames[SLOT_LOW], frames[SLOT_NOISE] = low_and_noise()
    frames[SLOT_FLAT] = 128
    frames[SLOT_SWEEP] = angle_sweep_frame()
    frames[255] = frames[0]
    one = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=1)
    single = [one(frames[s]) for s in range(256)]
    return frames, single, ORBextractor(1000, 1.2, 8, 20, 7, max_batch=256)


def test_headline_handle_256_frames(oracle, headline):
    from swarmmap_b200.orb import ORBextractor
    frames, single, prod = headline
    dbg = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=256, debug_score=True)
    k1, d1, n1 = prod.extract_batch(frames)
    k1, d1, n1 = k1.copy(), d1.copy(), n1.copy()
    k2, d2, n2 = prod.extract_batch(frames)  # second run
    kd, dd, nd = dbg.extract_batch(frames)   # pass 1 with the score map
    np.testing.assert_array_equal(n1, n2)
    np.testing.assert_array_equal(n1, nd)
    assert n1[SLOT_FLAT] == 0
    total = {}
    for s in range(256):
        r = _rows(k1, d1, n1, s)
        assert _same(r, _rows(k2, d2, n2, s)), f"slot {s}: second run differs"
        assert _same(r, _rows(kd, dd, nd, s)), f"slot {s}: debug-map handle differs"
        assert _same(r, single[s]), f"slot {s}: differs from the single-frame handle"
        orb_ref.merge(total, orb_ref.check_extractor_frame(dbg, s, *r, what=f"slot {s}"))
    assert _same(_rows(k1, d1, n1, 0), _rows(k1, d1, n1, 255))
    _report(total, "256-frame call")
    assert total["max_angle_err_rad"] <= orb_ref.ANGLE_TOL_RAD
    # rotation coverage of the sweep frame
    bins = np.unique(np.floor(kd[SLOT_SWEEP, :nd[SLOT_SWEEP]]["angle"]).astype(np.int64) % 360)
    print(f"angle sweep: {len(bins)} of 360 one-degree bins")
    assert len(bins) >= 300, len(bins)
    cpu = oracle.Extractor(1000, 1.2, 8, 20, 7)
    for s in (0, 255, SLOT_LOW, SLOT_NOISE, SLOT_SWEEP):
        _check_frame(dbg, cpu, frames[s], s, _rows(kd, dd, nd, s))


# batch -> level-0 row blocks of the pyramid walk on a 148-SM B200 at 752x480 (extract.cu enqueue): 8 rows below
# 4 frames, at least 16 from 4, 32 at 64 and the 64-row cap from about 150 frames; the pass-2 grid grows with the batch
@pytest.mark.parametrize("batch", [1, 3, 4, 17, 64, 200],
                         ids=["1-frame-8row", "3-frame-8row", "4-frame-16row", "17-frame-16row", "64-frame-32row",
                              "200-frame-64row"])
def test_partial_calls_on_headline_handle(headline, batch):
    """Smaller calls on the handle the 256-frame call used (nothing of a larger call may leak into a smaller one)."""
    frames, single, ex = headline
    first = 256 - batch if batch > 1 else SLOT_LOW  # the tail holds the noise, flat and sweep slots for batch >= 64
    k, d, n = ex.extract_batch(frames[first:first + batch])
    for s in range(batch):
        assert _same(_rows(k, d, n, s), single[first + s]), f"batch {batch}: frame {first + s} differs"


@pytest.mark.parametrize("nf,batch", [(2000, 50), (4000, 100)])
def test_kitti_handles(oracle, swm, nf, batch):
    """bench.py's KITTI-shaped handles: 50-frame calls at 2000 features and 100-frame calls at 4000 features."""
    from swarmmap_b200.orb import ORBextractor
    seq = synth.make_sequence(100, 1241, 376, 20220405)[:batch]
    ex = ORBextractor(nf, 1.2, 8, 20, 7, max_batch=batch, debug_score=True)
    one = ORBextractor(nf, 1.2, 8, 20, 7, max_batch=1)
    k, d, n = ex.extract_batch(seq)
    total = {}
    for s in range(batch):
        r = _rows(k, d, n, s)
        assert _same(r, one(seq[s])), f"frame {s} differs from the single-frame handle"
        orb_ref.merge(total, orb_ref.check_extractor_frame(ex, s, *r, what=f"frame {s}"))
    _report(total, f"{nf} features x {batch} frames")
    cpu = oracle.Extractor(nf, 1.2, 8, 20, 7)
    for s in (0, batch // 2, batch - 1):
        _check_frame(ex, cpu, seq[s], s, _rows(k, d, n, s))


def test_fast_run_edges(oracle, swm):
    """1 tile per warp (max_batch 7) and 4 (max_batch 8) give the same bytes; then the retry-heavy frames at widths
    whose level-0 rows hold 22, 23, 24 and 25 tiles, so that the last 4-tile run of a row holds 2, 3, 4 and 1."""
    from swarmmap_b200.orb import ORBextractor
    frames = synth.make_batch(7, W, H, 20220413)
    frames[2], frames[5] = low_and_noise()
    e7 = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=7)
    e8 = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=8, debug_score=True)
    a = e7.extract_batch(frames)
    b = e8.extract_batch(frames)
    for s in range(7):
        assert _same(_rows(*a, s), _rows(*b, s)), f"slot {s}: 1 vs 4 tiles per warp"
    cpu = oracle.Extractor(1000, 1.2, 8, 20, 7)
    for w in (736, 752, 800, 832):
        low, noise = low_and_noise(w, H)
        batch = synth.make_batch(8, w, H, 20220414)
        batch[3], batch[6] = low, noise
        k, d, n = e8.extract_batch(batch)
        for s, img in ((3, low), (6, noise)):
            _check_frame(e8, cpu, img, s, _rows(k, d, n, s))
