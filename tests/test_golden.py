"""Committed golden fixtures (tests/golden/, produced by make_golden.py from the oracle).
CPU: the oracle still reproduces them (guards the checker itself).  GPU: the CUDA path reproduces
them without the oracle in the loop."""
import hashlib
import os

import numpy as np
import pytest

import orb_ref
from swarmmap_b200 import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _load(name):
    return np.load(os.path.join(GOLD, name))


@pytest.mark.parametrize("name", ["extract_euroc.npz", "extract_kitti.npz"])
def test_oracle_reproduces_extract_golden(oracle, name):
    g = _load(name)
    img = synth.make_frame(int(g["w"]), int(g["h"]), int(g["seed"]))
    assert sha(img) == str(g["frame_sha"]), "synthetic generator drifted"
    ex = oracle.Extractor(int(g["nfeatures"]), 1.2, 8, 20, 7)
    kps, desc = ex(img)
    assert kps.tobytes() == g["kps"].tobytes()
    np.testing.assert_array_equal(desc, g["desc"])
    for l in range(8):
        assert sha(ex.level(l, 0)) == str(g[f"plane_sha_{l}"])
        assert sha(ex.level(l, 1)) == str(g[f"blur_sha_{l}"])
        assert len(ex.level_fast(l)) == int(g[f"fast_count_{l}"])


def test_oracle_reproduces_match_golden(oracle):
    from swarmmap_b200.matcher import Frame
    g = _load("match_init.npz")
    seq = synth.make_sequence(4, 1241, 376, 20220405)
    assert sha(seq) == str(g["seq_sha"])
    ex = oracle.Extractor(4000, 1.2, 8, 20, 7)
    sf = oracle.scale_tables(1.2, 8)[0]
    fs = [Frame.from_keypoints(*ex(img), 1241, 376, sf) for img in seq]
    assert [f.N for f in fs] == g["n_kp"].tolist()
    prev = np.stack([fs[0].x, fs[0].y], 1).astype(np.float32)
    for k in (1, 2, 3):
        n, m12, prev = oracle.search_for_initialization(fs[0], fs[k], prev, 100, 0.9, True)
        assert n == int(g[f"n_{k}"])
        np.testing.assert_array_equal(m12, g[f"m12_{k}"])
        np.testing.assert_array_equal(prev, g[f"prev_{k}"])


def test_oracle_reproduces_cv2_undistort_golden(oracle):
    """undistort_cv2.npz holds cv2.undistortPoints outputs (OpenCV is the third-party reference behind
    Frame::UndistortKeyPoints): the oracle equals them bit for bit, without cv2 in the loop."""
    g = _load("undistort_cv2.npz")
    for name in ("euroc", "tum1"):
        np.testing.assert_array_equal(oracle.undistort_points(g["xy"], g[f"cam_{name}"]), g[f"und_{name}"])
        m = g[f"und_{name}"][-4:]
        exp = [min(m[0, 0], m[2, 0]), max(m[1, 0], m[3, 0]), min(m[0, 1], m[1, 1]), max(m[2, 1], m[3, 1])]
        np.testing.assert_array_equal(oracle.image_bounds(752, 480, g[f"cam_{name}"]), np.array(exp, np.float32))


def _next_rows():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return mg


def test_oracle_reproduces_next_rows_golden(oracle):
    g = _load("next_rows.npz")
    mg = _next_rows()
    i = mg.next_rows_inputs()
    assert sha(i["seq"]) == str(g["seq_sha"]) and sha(np.frombuffer(i["blob"], np.uint8)) == str(g["vocab_sha"])
    out = mg.next_rows_outputs(i)
    for k, v in out.items():
        np.testing.assert_array_equal(np.asarray(v), g[k], err_msg=k)


@pytest.mark.gpu
def test_gpu_reproduces_next_rows_golden(swm):
    """The CUDA path against the committed outputs, no oracle in the loop."""
    from swarmmap_b200.bow import ORBVocabulary
    from swarmmap_b200.matcher import Frame, ORBmatcher
    from swarmmap_b200.orb import ORBextractor
    g = _load("next_rows.npz")
    seq = synth.make_sequence(2, 752, 480, 20220406)
    assert sha(seq) == str(g["seq_sha"])
    ex = ORBextractor(1000, 1.2, 8, 20, 7)
    sf = ex.GetScaleFactors()
    fs = [Frame.from_keypoints(*ex(img), 752, 480, sf) for img in seq]
    blob = synth.make_vocabulary(10, 3, seed=42)
    r = ORBVocabulary(blob).transform(fs[0].desc, 2)
    np.testing.assert_array_equal(r.word_ids, g["bow_words"])
    np.testing.assert_array_equal(r.values, g["bow_values"])
    np.testing.assert_array_equal(r.node_ids, g["bow_nodes"])
    np.testing.assert_array_equal(r.feats, g["bow_feats"])
    rng = np.random.default_rng(17)
    from swarmmap_b200.matcher import FeatureVector
    node = lambda f: (f.desc[:, 0].astype(np.int64) * 7 + f.desc[:, 5]) % 40
    fv = [FeatureVector(node(f)) for f in fs]
    v1 = (rng.random(fs[0].N) < 0.7).astype(np.uint8)
    v2 = (rng.random(fs[1].N) < 0.8).astype(np.uint8)
    K = np.array([[458.654, 0, 367.215], [0, 457.296, 248.375], [0, 0, 1]])
    t = np.array([0.3, 0.05, 0.02])
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    F12 = (np.linalg.inv(K).T @ tx @ np.linalg.inv(K)).astype(np.float32)
    s2 = (sf * sf).astype(np.float32)
    m = ORBmatcher(0.6, True)
    tn, tm = m.SearchForTriangulation(fs[0], fv[0], v1, fs[1], fv[1], v2, F12, 400.0, 200.0, sf, s2)
    assert tn == int(g["tri_n"])
    np.testing.assert_array_equal(tm, g["tri_matches"])
    u = (fs[0].x + rng.normal(0, 1.5, fs[0].N)).astype(np.float32)
    v = (fs[0].y + rng.normal(0, 1.5, fs[0].N)).astype(np.float32)
    pred = np.clip(fs[0].octave + rng.integers(-1, 2, fs[0].N), 0, 7).astype(np.int32)
    radius = (np.float32(12.0) * sf[pred]).astype(np.float32)
    inv_s2 = (np.float32(1.0) / s2).astype(np.float32)
    bi, bd = m.window_best(fs[1], fs[0].desc, u, v, radius, pred, np.ones(fs[0].N, np.uint8), inv_s2, 5.99)
    np.testing.assert_array_equal(bi, g["best_idx"])
    np.testing.assert_array_equal(bd, g["best_dist"])
    sizes = [1, 2, 3, 8, 0, 31, 64]
    obs = np.concatenate([fs[0].desc[:20], fs[1].desc[:89]])[:sum(sizes)]
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    db, dm = m.ComputeDistinctiveDescriptors(obs, offsets)
    np.testing.assert_array_equal(db, g["distinct_idx"])
    np.testing.assert_array_equal(dm, g["distinct_median"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["extract_euroc.npz", "extract_kitti.npz"])
def test_gpu_reproduces_extract_golden(swm, name):
    from swarmmap_b200.orb import ORBextractor
    g = _load(name)
    img = synth.make_frame(int(g["w"]), int(g["h"]), int(g["seed"]))
    ex = ORBextractor(int(g["nfeatures"]), 1.2, 8, 20, 7)
    kps, desc = ex(img)
    gk = g["kps"]
    assert len(kps) == len(gk)
    for f in ("x", "y", "size", "response", "octave", "class_id"):
        np.testing.assert_array_equal(kps[f], gk[f])
    d = np.abs(kps["angle"] - gk["angle"])
    assert np.deg2rad(np.minimum(d, 360 - d).max()) <= 1e-4
    agree = 1.0 - np.unpackbits(desc ^ g["desc"]).sum() / float(desc.size * 8)
    assert agree >= 0.999
    for l in range(8):
        assert sha(ex.debug_plane(0, l, 0)) == str(g[f"plane_sha_{l}"])
        assert sha(ex.debug_plane(0, l, 1)) == str(g[f"blur_sha_{l}"])
        assert min(len(ex.debug_points(0, l, 0)), 10000) == int(g[f"fast_count_{l}"])
    orb_ref.check_extractor_frame(ex, 0, kps, desc, score=False, what=name)


@pytest.mark.gpu
def test_gpu_extract_then_match_golden(swm):
    """extract (GPU) -> SearchForInitialization (GPU) end to end against the golden match indices.
    Descriptors may differ from the oracle's in <0.1 % of bits, so allow a handful of match flips."""
    from swarmmap_b200.matcher import Frame, ORBmatcher
    from swarmmap_b200.orb import ORBextractor
    g = _load("match_init.npz")
    seq = synth.make_sequence(4, 1241, 376, 20220405)
    ex = ORBextractor(4000, 1.2, 8, 20, 7)
    fs = [Frame.from_keypoints(*ex(img), 1241, 376) for img in seq]
    assert [f.N for f in fs] == g["n_kp"].tolist()
    m = ORBmatcher(0.9, True)
    prev = np.stack([fs[0].x, fs[0].y], 1).astype(np.float32).copy()
    for k in (1, 2, 3):
        n, m12 = m.SearchForInitialization(fs[0], fs[k], prev, 100)
        same = (m12 == g[f"m12_{k}"]).mean()
        assert same >= 0.995 and abs(n - int(g[f"n_{k}"])) <= 5, (k, n, int(g[f"n_{k}"]), same)
        prev = g[f"prev_{k}"].copy()
