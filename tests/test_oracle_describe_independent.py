"""Independent numpy reading of the orientation and descriptor stages (reference code/src/cuda/Fast_gpu.cu:403-456
IC_Angle_kernel, code/src/cuda/Orb_gpu.cu:63-104 calcOrb_kernel) against the oracle's orc_extract output, for the
octave-0 keypoints of a frame (their coordinates are level coordinates).  The un-blurred and blurred level planes the
stages read are the ones tests/test_oracle_cv2.py pins to cv2."""
import numpy as np

from orb_ref import load_pattern
from swarmmap_b200 import synth


def test_ic_angle_and_rbrief_vs_numpy(oracle):
    img = synth.make_frame(640, 400, 123)
    ex = oracle.Extractor(600, 1.2, 8, 20, 7)
    kps, desc = ex(img)
    plain = ex.level(0, 0).astype(np.int64)   # bordered (19 px) un-blurred level 0
    blur = ex.level(0, 1)                     # blurred ROI
    blur_b = np.pad(blur, 19, mode="reflect").astype(np.int64)  # reads stay inside the ROI; the pad only keeps indexing simple
    umax = oracle.umax()
    pat = load_pattern()
    idx = np.nonzero(kps["octave"] == 0)[0][:150]
    assert len(idx) > 50
    max_dang, bit_err, bits = 0.0, 0, 0
    for i in idx:
        x, y = int(kps["x"][i]), int(kps["y"][i])
        cx, cy = x + 19, y + 19
        m10 = sum(u * plain[cy, cx + u] for u in range(-15, 16))
        m01 = 0
        for v in range(1, 16):
            d = int(umax[v])
            us = np.arange(-d, d + 1)
            plus, minus = plain[cy + v, cx + us], plain[cy - v, cx + us]
            m01 += v * int((plus - minus).sum())
            m10 += int((us * (plus + minus)).sum())
        ang = np.float32(np.arctan2(np.float32(m01), np.float32(m10)))
        if ang < 0:
            ang = np.float32(ang + np.float32(2.0) * np.float32(np.pi))
        ang_deg = np.float32(ang * (np.float32(180.0) / np.float32(np.pi)))
        dang = abs(float(ang_deg) - float(kps["angle"][i]))
        max_dang = max(max_dang, min(dang, 360 - dang))
        # descriptor from the oracle's own angle (so that an ulp of atan2 cannot flip a rounding)
        a_rad = np.float32(kps["angle"][i]) * np.float32(np.pi / 180.0)
        a, b = np.float32(np.cos(a_rad)), np.float32(np.sin(a_rad))
        px, py = pat[:, 0].astype(np.float32), pat[:, 1].astype(np.float32)
        ry = np.rint((px * b).astype(np.float32) + (py * a).astype(np.float32)).astype(np.int64)   # __float2int_rn
        rx = np.rint((px * a).astype(np.float32) - (py * b).astype(np.float32)).astype(np.int64)
        vals = blur_b[cy + ry, cx + rx]
        bitsv = (vals[0::2] < vals[1::2]).astype(np.uint8)
        exp = np.packbits(bitsv, bitorder="little")
        bit_err += int(np.unpackbits(exp ^ desc[i]).sum())
        bits += 256
    assert np.deg2rad(max_dang) <= 1e-4, max_dang       # north_star's orientation tolerance
    assert bit_err / bits <= 1e-3, (bit_err, bits)       # and its descriptor-bit tolerance (cos/sin ulp near .5 roundings)
