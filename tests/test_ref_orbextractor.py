"""The oracle against the REFERENCE's own ORBextractor.cc, compiled unmodified (make -C oracle ref ->
oracle/_ref/liborbextractor_ref.so; OpenCV headers are stand-ins from oracle/ref_shim, the CUDA helper classes are
stubs).  Exercised: the constructor (scale / sigma tables, per-level quotas, umax, the rBRIEF pattern it uploads) and
ORBextractor::DistributeOctTree with ExtractorNode::DivideNode -- the most intricate stage of the extractor.

The reference orders equal-sized quadtree nodes by std::sort on pair<int, ExtractorNode*>, i.e. by the ADDRESS of
std::list nodes; with glibc malloc freed nodes are recycled, so that order depends on allocator internals.  The
oracle freezes the tie as "later-created node first".  With a non-recycling allocator (addresses grow with creation
order) the reference's own code realises exactly that definition: selection AND order must then be identical.  With
the stock allocator only the tie-dependent part may differ."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "liborbextractor_ref.so")
pytestmark = pytest.mark.skipif(not os.path.exists(LIB), reason="needs oracle/_ref/liborbextractor_ref.so, compiled by `make -C oracle ref` "
                                                                "from the reference project's sources, which the repository does not contain")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def ref():
    L = C.CDLL(LIB)
    L.ref_orb_create.restype = C.c_void_p
    L.ref_orb_create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
    L.ref_orb_destroy.argtypes = [C.c_void_p]
    L.ref_orb_tables.argtypes = [C.c_void_p] * 8
    L.ref_orb_distribute.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 7 + [C.c_void_p, C.c_int, C.c_int]
    return L


@pytest.mark.parametrize("nfeatures,scale,nlevels", [(1000, 1.2, 8), (2000, 1.2, 8), (4000, 1.2, 8), (500, 1.2, 8),
                                                     (1500, 1.1, 12), (800, 1.5, 5), (3000, 1.3, 6)])
def test_constructor_tables_equal_reference(oracle, ref, nfeatures, scale, nlevels):
    e = ref.ref_orb_create(nfeatures, scale, nlevels, 20, 7)
    sf, isf, s2, is2 = [np.zeros(nlevels, np.float32) for _ in range(4)]
    q = np.zeros(nlevels, np.int32)
    um = np.zeros(16, np.int32)
    pat = np.zeros(1024, np.int8)
    ref.ref_orb_tables(e, _p(sf), _p(isf), _p(s2), _p(is2), _p(q), _p(um), _p(pat))
    ref.ref_orb_destroy(e)
    for a, b in zip((sf, isf, s2, is2), oracle.scale_tables(scale, nlevels)):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(q, oracle.level_quotas(nfeatures, scale, nlevels))
    np.testing.assert_array_equal(um, oracle.umax())
    txt = open(os.path.join(ROOT, "oracle", "orb_pattern_data.inc")).read()
    vals = np.array([int(v) for v in re.findall(r"-?\d+", txt[txt.index("{") + 1:txt.index("};")])], np.int8)
    np.testing.assert_array_equal(pat, vals)  # bit_pattern_31_ as the reference hands it to the GPU


def _case(rng, trial):
    W, H = int(rng.integers(40, 1300)), int(rng.integers(40, 600))
    if not 1 <= round(W / H) <= 16:
        return None
    n = int(rng.integers(0, 3000)) if trial % 4 else int(rng.integers(0, 30))
    N = int(rng.integers(1, 1100)) if trial % 5 else int(rng.integers(0, 20))
    if trial % 4 == 2:  # clustered points
        cx, cy = rng.integers(3, W - 3, 5), rng.integers(3, H - 3, 5)
        xs = np.clip((cx[rng.integers(0, 5, n)] + rng.normal(0, 20, n)).astype(int), 3, W - 4)
        ys = np.clip((cy[rng.integers(0, 5, n)] + rng.normal(0, 20, n)).astype(int), 3, H - 4)
    else:
        xs, ys = rng.integers(3, W - 3, n), rng.integers(3, H - 3, n)
    key = np.unique(ys.astype(np.int64) * 4096 + xs)  # distinct pixels, raster order (how FAST delivers them)
    ys, xs = (key // 4096).astype(np.int16), (key % 4096).astype(np.int16)
    sc = rng.integers(7, 40 if trial % 4 == 3 else 256, len(key)).astype(np.int32)  # many response ties
    return W, H, N, xs, ys, sc


def _both(oracle, ref, e, W, H, N, xs, ys, sc, monotonic):
    pts = np.zeros(len(xs), oracle.FASTPT_DTYPE)
    pts["x"], pts["y"], pts["score"] = xs, ys, sc
    o = oracle.octree(pts, 16, 16 + W, 16, 16 + H, N)
    inp = np.ascontiguousarray(np.stack([xs, ys, sc], 1).astype(np.float32)).reshape(-1, 3)
    out = np.zeros((len(xs) + 16, 3), np.float32)
    m = ref.ref_orb_distribute(e, _p(inp), len(xs), 16, 16 + W, 16, 16 + H, N, 0, _p(out), len(out), int(monotonic))
    return o, out[:m].astype(np.int64)


def test_distribute_octtree_equals_reference_code(oracle, ref):
    """Non-recycling allocator: the reference's DistributeOctTree == the oracle, selection and order, on random,
    clustered, tie-heavy, tiny and over-provisioned inputs."""
    e = ref.ref_orb_create(1000, 1.2, 8, 20, 7)
    rng = np.random.default_rng(5)
    done = 0
    for trial in range(400):
        c = _case(rng, trial)
        if c is None:
            continue
        o, r = _both(oracle, ref, e, *c, monotonic=True)
        assert len(o) == len(r), trial
        np.testing.assert_array_equal(r[:, 0], o["x"], err_msg=f"trial {trial}")
        np.testing.assert_array_equal(r[:, 1], o["y"], err_msg=f"trial {trial}")
        np.testing.assert_array_equal(r[:, 2], o["score"], err_msg=f"trial {trial}")
        done += 1
    ref.ref_orb_destroy(e)
    assert done > 300


def test_distribute_octtree_on_real_fast_candidates(oracle, ref):
    """The per-level FAST candidates of a real (synthetic) frame with the extractor's own quotas."""
    from swarmmap_b200 import synth
    e = ref.ref_orb_create(1000, 1.2, 8, 20, 7)
    img = synth.make_frame(752, 480, 20220404)
    ex = oracle.Extractor(1000, 1.2, 8, 20, 7)
    ex(img)
    ws, hs = oracle.level_sizes(752, 480)
    quotas = oracle.level_quotas(1000)
    for l in range(8):
        cand = ex.level_fast(l)
        W, H = int(ws[l]) - 32, int(hs[l]) - 32
        o, r = _both(oracle, ref, e, W, H, int(quotas[l]), cand["x"], cand["y"], cand["score"], monotonic=True)
        assert len(o) == len(r) and len(o) > 0
        np.testing.assert_array_equal(r[:, 0], o["x"])
        np.testing.assert_array_equal(r[:, 1], o["y"])
        np.testing.assert_array_equal(r[:, 2], o["score"])
    ref.ref_orb_destroy(e)


def test_stock_allocator_differs_only_in_ties(oracle, ref):
    """With glibc malloc the reference's address-ordered ties are allocator-dependent: the counts agree to within the
    overshoot of one split and the selections overlap almost completely; where no equal-size tie can arise (every point gets its own node)
    the results are identical."""
    e = ref.ref_orb_create(1000, 1.2, 8, 20, 7)
    rng = np.random.default_rng(11)
    overlaps = []
    for trial in range(120):
        c = _case(rng, trial)
        if c is None:
            continue
        o, r = _both(oracle, ref, e, *c, monotonic=False)
        assert abs(len(o) - len(r)) <= 8  # which nodes are split last decides by how much the loop overshoots N
        a = set(zip(o["x"].tolist(), o["y"].tolist()))
        b = set(map(tuple, r[:, :2].tolist()))
        if len(a):
            overlaps.append(len(a & b) / len(a))
        if c[2] >= len(c[3]) * 4 and len(a):  # N far above the number of points: no "largest first" phase
            assert a == b
    ref.ref_orb_destroy(e)
    assert np.mean(overlaps) > 0.95  # measured here: 0.99 (bounds kept loose: they depend on the C library's malloc)
