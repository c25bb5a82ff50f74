"""The oracle's DBoW2 restatement against the REFERENCE's own DBoW2, compiled unmodified from
/root/reference/code/Thirdparty/DBoW2 by `make -C oracle ref` (against oracle/ref_shim's stand-in for
opencv2/core/core.hpp) into oracle/_ref/libdbow2_ref.so.  This pins the SURVEY section 8(f) rank-2 row (and
DescriptorDistance's bit count) to the reference itself: word ids, TF-IDF values as bit-exact doubles, FeatureVector
nodes and feature lists.  Skipped when the library has not been built (it needs /root/reference at build time; the
built file travels to the GPU box with the other .so files)."""
import ctypes as C
import os

import numpy as np
import pytest

from swarmmap_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libdbow2_ref.so")
pytestmark = pytest.mark.skipif(not os.path.exists(LIB), reason="needs oracle/_ref/libdbow2_ref.so, compiled by `make -C oracle ref` "
                                                                "from the reference project's sources, which the repository does not contain")


@pytest.fixture(scope="module")
def ref():
    L = C.CDLL(LIB)
    L.ref_vocab_load.restype = C.c_void_p
    L.ref_vocab_load.argtypes = [C.c_char_p]
    L.ref_vocab_destroy.argtypes = [C.c_void_p]
    L.ref_vocab_info.argtypes = [C.c_void_p] * 4
    L.ref_bow_transform.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 6
    L.ref_forb_distance.argtypes = [C.c_void_p, C.c_void_p]
    L.ref_score.restype = C.c_double
    L.ref_score.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _ref_transform(L, h, desc, levelsup):
    desc = np.ascontiguousarray(desc, np.uint8)
    n = len(desc)
    wid = np.zeros(n + 1, np.uint32); wv = np.zeros(n + 1, np.float64)
    nid = np.zeros(n + 1, np.uint32); off = np.zeros(n + 2, np.int32); feats = np.zeros(n + 1, np.uint32)
    nn = C.c_int32(0)
    nw = L.ref_bow_transform(h, _p(desc), n, levelsup, _p(wid), _p(wv), _p(nid), _p(off), _p(feats), C.byref(nn))
    return wid[:nw], wv[:nw], nid[:nn.value], off[:nn.value + 1], feats[:off[nn.value]]


def _descriptors(blob, n, seed):
    rng = np.random.default_rng(seed)
    rec = np.frombuffer(blob[24:], np.dtype([("parent", "<i4"), ("desc", "u1", 32), ("weight", "<f4"), ("leaf", "u1")]))
    leaf = rec[rec["leaf"] == 1]["desc"]
    d = leaf[rng.integers(0, len(leaf), n)].copy()
    d[: n // 2, :6] ^= rng.integers(0, 256, (n // 2, 6), dtype=np.uint8)
    d[n // 2: n // 2 + n // 8] = rng.integers(0, 256, (n // 8, 32), dtype=np.uint8)
    return d


# levelsup such that L - levelsup <= the shallowest leaf (depth 1 with early leaves): a leaf above that level makes
# the reference read an uninitialised NodeId (TemplatedVocabulary.h:1175 / :1250-1276), which has no defined answer
@pytest.mark.parametrize("k,L,levelsup,early", [(10, 3, 2, 0.03), (10, 4, 2, 0.0), (10, 4, 4, 0.03), (7, 5, 4, 0.05), (4, 2, 1, 0.1)])
@pytest.mark.parametrize("weighting,scoring", [(0, 0), (1, 1), (2, 0), (3, 5), (0, 5)])
def test_oracle_transform_equals_reference_dbow2(oracle, ref, tmp_path, k, L, levelsup, early, weighting, scoring):
    blob = synth.make_vocabulary(k, L, seed=100 * k + L, early_leaf=early, zero_weight=0.05, weighting=weighting,
                                 scoring=scoring)
    path = tmp_path / "voc.bin"
    path.write_bytes(blob)
    h = ref.ref_vocab_load(str(path).encode())
    assert h
    try:
        o = oracle.Vocabulary(blob)
        info = [C.c_int32() for _ in range(3)]
        ref.ref_vocab_info(h, *[C.byref(x) for x in info])
        assert (info[0].value, info[1].value) == (o.k, o.L)
        # the reference's reader runs its loop once more at end-of-file and appends a copy of the last node
        # (TemplatedVocabulary.h:1493-1516); the copy never wins a strict '<' against its twin
        assert info[2].value in (o.n_words, o.n_words + 1)
        for n in (1, 50, 1500):
            d = _descriptors(blob, n, n)
            got = o.transform(d, levelsup)
            exp = _ref_transform(ref, h, d, levelsup)
            for a, b, name in zip(got, exp, ("word ids", "word values", "node ids", "offsets", "features")):
                np.testing.assert_array_equal(a, b, err_msg=name)
    finally:
        ref.ref_vocab_destroy(h)


def test_descriptor_distance_equals_forb_distance(oracle, ref):
    rng = np.random.default_rng(0)
    a = rng.integers(0, 256, (500, 32), dtype=np.uint8)
    b = rng.integers(0, 256, (500, 32), dtype=np.uint8)
    b[:50] = a[:50]
    b[50:60] = ~a[50:60]
    for i in range(500):
        d = ref.ref_forb_distance(_p(a[i]), _p(b[i]))
        assert d == int(np.unpackbits(a[i] ^ b[i]).sum()) == oracle.hamming256(a[i], b[i])


def test_reference_l1_score_of_oracle_vectors(oracle, ref, tmp_path):
    """The BowVectors the oracle produces are what the reference's KeyFrameDatabase scoring expects: L1-normalised,
    score(v, v) = 1, score of disjoint vectors = 0."""
    blob = synth.make_vocabulary(10, 3, seed=9)
    path = tmp_path / "voc.bin"
    path.write_bytes(blob)
    h = ref.ref_vocab_load(str(path).encode())
    o = oracle.Vocabulary(blob)
    d = _descriptors(blob, 800, 1)
    w, wv, *_ = o.transform(d, 2)
    w = np.ascontiguousarray(w, np.uint32); wv = np.ascontiguousarray(wv, np.float64)
    assert abs(ref.ref_score(h, _p(w), _p(wv), len(w), _p(w), _p(wv), len(w)) - 1.0) < 1e-9
    w2 = (w + np.uint32(10 ** 6)).astype(np.uint32)
    assert abs(ref.ref_score(h, _p(w), _p(wv), len(w), _p(w2), _p(wv), len(w))) < 1e-12
    ref.ref_vocab_destroy(h)
