"""The single matcher calls (swm_match_window / _init / _bow and their _resident forms) check their arguments as the
batch entry points check a job: for each input below, the single call and a one-job batch must return the same code.
The cases are invalid input that the single calls once accepted or dereferenced: a negative SearchForInitialization
window, a resident target that was created but never built, FeatureVector node ids out of order or repeated, NULL
FeatureVector arrays, and a ratio mode other than 0 / 1."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

E_INVALID, E_STATE = -1, -5


def _frame(rng, n=300, w=640, h=480):
    from swarmmap_b200.matcher import Frame
    return Frame(rng.uniform(0, w, n), rng.uniform(0, h, n), rng.integers(0, 4, n), rng.uniform(0, 360, n),
                 rng.integers(0, 256, (n, 32), dtype=np.uint8), (0.0, 0.0, float(w), float(h)))


@pytest.fixture(scope="module")
def setup(swm):
    from swarmmap_b200.matcher import ORBmatcher, ResidentFrame
    rng = np.random.default_rng(3)
    f1, f2 = _frame(rng), _frame(rng)
    return dict(lib=swm.load(), m=ORBmatcher(0.9, True), f1=f1, f2=f2, r1=ResidentFrame().upload(f1),
                r2=ResidentFrame().upload(f2), unbuilt=ResidentFrame())


def _operands(s, kind, tgt=None):
    """(host view or None, resident handle or None) of f1 and f2 (f2 replaced by `tgt` when given)."""
    if kind == "host":
        v1, v2 = s["f1"].view(), s["f2"].view()
        return (v1, None), (v2, None)
    return (None, s["r1"]._h), (None, (tgt or s["r2"])._h)


def _ref(x):
    return C.byref(x) if x is not None else None


def _init_rcs(s, kind, window, tgt=None):
    """Return codes of swm_match_init[_resident] and of swm_match_init_batch with one job, same arguments."""
    from swarmmap_b200._lib import InitJob, ptr
    lib, m = s["lib"], s["m"]
    (h1, d1), (h2, d2) = _operands(s, kind, tgt)
    n1 = s["f1"].N
    prev = np.stack([s["f1"].x, s["f1"].y], 1).astype(np.float32)
    out = np.full(n1, -1, np.int32)
    n = C.c_int(0)
    if kind == "host":
        rc1 = lib.swm_match_init(m._h, _ref(h1), _ref(h2), ptr(prev), ptr(out), window, 0.9, 1, C.byref(n))
    else:
        rc1 = lib.swm_match_init_resident(m._h, d1, d2, ptr(prev), ptr(out), window, 0.9, 1, C.byref(n))
    job = InitJob(C.addressof(h1) if h1 is not None else None, C.addressof(h2) if h2 is not None else None, d1, d2,
                  ptr(prev).value, ptr(out).value, window, 0.9, 1, 0)
    rc2 = lib.swm_match_init_batch(m._h, C.byref(job), 1)
    return rc1, rc2


def _window_rcs(s, kind, ratio_mode, tgt=None):
    """Return codes of swm_match_window[_resident] and of swm_match_window_batch with one job."""
    from swarmmap_b200._lib import WindowJob, WindowQuery, ptr
    lib, m, src = s["lib"], s["m"], s["f1"]
    (_, _), (h2, d2) = _operands(s, kind, tgt)
    mq = src.N
    radius = np.full(mq, 20.0, np.float32)
    lo, hi = src.octave - 1, src.octave + 1
    ones = np.ones(mq, np.uint8)
    q = WindowQuery(mq, ptr(src.desc).value, ptr(src.x).value, ptr(src.y).value, ptr(radius).value, ptr(lo).value,
                    ptr(hi).value, ptr(ones).value, ptr(src.angle).value, ptr(ones).value)
    asg = np.full(s["f2"].N, -1, np.int32)
    n = C.c_int(0)
    if kind == "host":
        rc1 = lib.swm_match_window(m._h, _ref(h2), C.byref(q), None, 100, ratio_mode, 0.9, 1, ptr(asg), C.byref(n))
    else:
        rc1 = lib.swm_match_window_resident(m._h, d2, C.byref(q), None, 100, ratio_mode, 0.9, 1, ptr(asg),
                                            C.byref(n))
    job = WindowJob(C.addressof(h2) if h2 is not None else None, d2, C.addressof(q), None, 100, ratio_mode, 0.9, 1,
                    ptr(asg).value, 0)
    rc2 = lib.swm_match_window_batch(m._h, C.byref(job), 1)
    return rc1, rc2


def _bow_rcs(s, kind, mode, fv1, fv2):
    """Return codes of swm_match_bow[_resident] and of swm_match_bow_batch with one job."""
    from swarmmap_b200._lib import BowJob, ptr
    lib, m = s["lib"], s["m"]
    (h1, d1), (h2, d2) = _operands(s, kind)
    v1 = np.ones(s["f1"].N, np.uint8)
    v2 = np.ones(s["f2"].N, np.uint8) if mode == 1 else None
    out = np.full(s["f2"].N if mode == 0 else s["f1"].N, -1, np.int32)
    n = C.c_int(0)
    p2 = ptr(v2) if v2 is not None else None
    if kind == "host":
        rc1 = lib.swm_match_bow(m._h, _ref(h1), C.byref(fv1), ptr(v1), _ref(h2), C.byref(fv2), p2, mode, 0.75, 1,
                                ptr(out), C.byref(n))
    else:
        rc1 = lib.swm_match_bow_resident(m._h, d1, C.byref(fv1), ptr(v1), d2, C.byref(fv2), p2, mode, 0.75, 1,
                                         ptr(out), C.byref(n))
    job = BowJob(C.addressof(h1) if h1 is not None else None, C.addressof(h2) if h2 is not None else None, d1, d2,
                 C.addressof(fv1), C.addressof(fv2), ptr(v1).value, p2.value if p2 is not None else None, mode, 0.75,
                 1, ptr(out).value, 0)
    rc2 = lib.swm_match_bow_batch(m._h, C.byref(job), 1)
    return rc1, rc2


def _featvec(frame, node_ids=None):
    """The frame's FeatureVector over 8 nodes; node_ids replaces the (ascending) ids when given."""
    from swarmmap_b200.matcher import FeatureVector
    fv = FeatureVector(np.arange(frame.N) % 8)
    if node_ids is not None:
        fv.node_ids = np.asarray(node_ids, np.uint32)
    return fv


@pytest.mark.parametrize("kind", ["host", "resident"])
def test_init_negative_window(setup, kind):
    assert _init_rcs(setup, kind, 10) == (0, 0)
    assert _init_rcs(setup, kind, -1) == (E_INVALID, E_INVALID)


def test_window_unbuilt_resident_target(setup):
    assert _window_rcs(setup, "resident", 0, tgt=setup["unbuilt"]) == (E_STATE, E_STATE)


def test_init_unbuilt_resident_target(setup):
    assert _init_rcs(setup, "resident", 10, tgt=setup["unbuilt"]) == (E_STATE, E_STATE)


@pytest.mark.parametrize("kind", ["host", "resident"])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("side", [1, 2])
def test_bow_node_ids_not_ascending(setup, kind, mode, side):
    good1, good2 = _featvec(setup["f1"]), _featvec(setup["f2"])
    assert _bow_rcs(setup, kind, mode, good1.view(), good2.view()) == (0, 0)
    for ids in ([0, 1, 2, 3, 5, 4, 6, 7], [0, 1, 2, 3, 3, 5, 6, 7]):  # swapped; repeated
        bad = _featvec(setup["f%d" % side], ids)
        fv1, fv2 = (bad, good2) if side == 1 else (good1, bad)
        assert _bow_rcs(setup, kind, mode, fv1.view(), fv2.view()) == (E_INVALID, E_INVALID), ids


@pytest.mark.parametrize("kind", ["host", "resident"])
@pytest.mark.parametrize("null", ["node_ids", "offsets", "feats"])
def test_bow_null_featvec_arrays(setup, kind, null):
    good1, good2 = _featvec(setup["f1"]), _featvec(setup["f2"])
    bad = good2.view()
    setattr(bad, null, None)
    assert _bow_rcs(setup, kind, 0, good1.view(), bad) == (E_INVALID, E_INVALID)


@pytest.mark.parametrize("kind", ["host", "resident"])
def test_window_ratio_mode_out_of_range(setup, kind):
    assert _window_rcs(setup, kind, 1) == (0, 0)
    for ratio_mode in (-1, 2):
        assert _window_rcs(setup, kind, ratio_mode) == (E_INVALID, E_INVALID), ratio_mode
