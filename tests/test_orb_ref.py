"""The per-keypoint float64 reference (tests/orb_ref.py) on the CPU oracle: it passes every keypoint of every octave
with no unexplained descriptor bit, and it catches wrong keypoints that the aggregate bar of the extractor tests
(>= 99.9 % of a frame's descriptor bits equal) lets through."""
import numpy as np
import pytest

import orb_ref
from swarmmap_b200 import synth

AGGREGATE_BAR = 0.999


def _frame(oracle, seed):
    ex = oracle.Extractor(1000, 1.2, 8, 20, 7)
    kps, desc = ex(synth.make_frame(752, 480, seed))
    planes = [ex.level(l, 0) for l in range(8)]
    blurs = [ex.level(l, 1) for l in range(8)]
    scores = [ex.level(l, 2) for l in range(8)]
    return kps, desc, planes, blurs, scores


def _agree(a, b):
    return 1.0 - np.unpackbits(a ^ b).sum() / float(a.size * 8)


def test_reference_tables_match_oracle(oracle):
    np.testing.assert_array_equal(orb_ref.UMAX, oracle.umax())
    assert orb_ref.PATTERN.shape == (512, 2) and np.abs(orb_ref.PATTERN).max() == 13


def test_oracle_passes_per_keypoint_reference(oracle):
    sf = oracle.scale_tables(1.2, 8)[0]
    total = {}
    for seed in (20220404, 11, 12):
        kps, desc, planes, blurs, scores = _frame(oracle, seed)
        assert set(np.unique(kps["octave"]).tolist()) == set(range(8))
        orb_ref.merge(total, orb_ref.check_keypoints(kps, desc, planes, blurs, sf, scores, what=f"seed {seed}"))
    print(f"oracle vs float64: {total['n']} keypoints, max angle error {total['max_angle_err_rad']:.2e} rad, "
          f"{total['ambiguous_bits']} ambiguous bits")
    assert total["max_angle_err_rad"] <= orb_ref.ANGLE_TOL_RAD


def test_mutations_caught(oracle):
    sf = oracle.scale_tables(1.2, 8)[0]
    kps, desc, planes, blurs, scores = _frame(oracle, 20220404)
    check = lambda k, d: orb_ref.check_keypoints(k, d, planes, blurs, sf, scores)
    check(kps, desc)

    # 1. one flipped bit, on a keypoint of octave 3
    i = int(np.nonzero(kps["octave"] == 3)[0][5])
    d1 = desc.copy()
    d1[i, 17] ^= 1 << 4
    assert _agree(d1, desc) >= AGGREGATE_BAR
    with pytest.raises(AssertionError, match=rf"keypoint {i} .*byte 17 bit 4"):
        check(kps, d1)

    # 2. two keypoints' descriptors swapped: the closest pair (>= 16 bits apart) keeps the aggregate above the bar
    dist = np.unpackbits(desc[:, None, :] ^ desc[None, :, :], axis=2).sum(2)
    dist[dist < 16] = 1 << 20
    a, b = np.unravel_index(int(np.argmin(dist)), dist.shape)
    d2 = desc.copy()
    d2[[a, b]] = d2[[b, a]]
    assert _agree(d2, desc) >= AGGREGATE_BAR
    with pytest.raises(AssertionError, match=rf"keypoint {min(a, b)} .*descriptor byte"):
        check(kps, d2)

    # 3. one angle moved by 0.05 degrees
    k3 = kps.copy()
    k3["angle"][i] = np.float32((float(k3["angle"][i]) + 0.05) % 360.0)
    with pytest.raises(AssertionError, match=rf"keypoint {i} .*angle"):
        check(k3, desc)

    # 4. one descriptor computed from the un-blurred plane instead of the blurred one
    o = int(kps["octave"][i])
    lx = np.array([int(np.rint(kps["x"][i] / sf[o]))])
    ly = np.array([int(np.rint(kps["y"][i] / sf[o]))])
    plain_roi = planes[o][orb_ref.EDGE:-orb_ref.EDGE, orb_ref.EDGE:-orb_ref.EDGE]
    bits, _ = orb_ref.ref_descriptors(plain_roi, lx, ly, kps["angle"][i:i + 1].astype(np.float64))
    d4 = desc.copy()
    d4[i] = np.packbits(bits[0], bitorder="little")
    assert (d4[i] != desc[i]).any()
    with pytest.raises(AssertionError, match=rf"keypoint {i} .*descriptor byte"):
        check(kps, d4)
