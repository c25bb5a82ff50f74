"""Latency of the single matcher calls against the same problem sent as a one-job batch, alternating the two forms call
by call in one process, with a check that both give the same output bit for bit.  Only the public Python API is used
(ORBmatcher.match_window / SearchForInitialization / SearchByBoW and their *Batch forms), so the same file runs against
any tree that has both forms.  Each call returns host results after a stream synchronise; the host clock around it is
the latency a caller sees, Python wrapper included.

Shapes: match_window (th 15, check_ori on) with 1000 sources into a 752x480 frame of ~1000 keypoints and with 4000
sources into a 1241x376 frame of ~4000 keypoints; SearchForInitialization on 4000-feature 1241x376 frames, window 100;
SearchByBoW mode 0 and mode 1 on 752x480 frames with a synthetic node_of_feature.  Each with host-array and resident
operands.  Writes one JSON file with the card's name and power limit, read in the same run.

  python tools/single_call_probe.py --out profiles/single_call_probe.json [--label parent] [--warmup 20] [--calls 300]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from swarmmap_b200 import synth  # noqa: E402
from swarmmap_b200.matcher import FeatureVector, Frame, ORBmatcher, ResidentFrame  # noqa: E402
from swarmmap_b200.orb import ORBextractor  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def frames(w, h, nfeat, seed, count=2):
    ex = ORBextractor(nfeat, 1.2, 8, 20, 7)
    sf = ex.GetScaleFactors()
    return [Frame.from_keypoints(*ex(img), w, h, sf) for img in synth.make_sequence(count, w, h, seed)]


def window_pair(m, src, tgt, tgt_op):
    """SearchByProjection(cur, last, 15)'s window query of `src`'s keypoints into `tgt`."""
    sf = np.asarray(tgt.mvScaleFactors, np.float32)
    kw = dict(tgt=tgt_op, desc=src.desc, u=src.x, v=src.y, radius=(np.float32(15) * sf[src.octave]).astype(np.float32),
              min_level=src.octave - 1, max_level=src.octave + 1, valid=np.ones(src.N, np.uint8),
              blocks=np.ones(src.N, np.uint8), th_dist=100, ratio_mode=0, angle=src.angle, check_ori=True)

    def single():
        return m.match_window(assignment=np.full(tgt.N, -1, np.int32), **kw)

    def batch():
        return m.match_window_batch([dict(kw, assignment=np.full(tgt.N, -1, np.int32))])[0]

    return single, batch


def init_pair(m, f1, op1, op2):
    prev0 = np.stack([f1.x, f1.y], 1).astype(np.float32)

    def single():
        prev = prev0.copy()
        n, m12 = m.SearchForInitialization(op1, op2, prev, 100)
        return n, m12, prev

    def batch():
        prev = prev0.copy()
        n, m12 = m.SearchForInitializationBatch([(op1, op2, prev)], 100)[0]
        return n, m12, prev

    return single, batch


def bow_pair(m, f1, f2, op1, op2, mode, rng):
    # synthetic vocabulary: the node of a feature is decided by its descriptor's first byte (64 nodes), so features
    # that match across the two frames mostly share a node, as they do under a real vocabulary
    fv1, fv2 = FeatureVector(f1.desc[:, 0] >> 2), FeatureVector(f2.desc[:, 0] >> 2)
    v1 = (rng.random(f1.N) < 0.6).astype(np.uint8)
    v2 = (rng.random(f2.N) < 0.6).astype(np.uint8) if mode == 1 else None

    def single():
        return m.SearchByBoW(op1, fv1, v1, op2, fv2, v2)

    def batch():
        return m.SearchByBoWBatch([(op1, fv1, v1, op2, fv2, v2)])[0]

    return single, batch


def same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


def measure(single, batch, warmup, calls):
    ts, tb, identical, first = [], [], True, None
    for i in range(warmup + calls):
        order = (("s", single), ("b", batch)) if i % 2 == 0 else (("b", batch), ("s", single))
        got = {}
        for key, fn in order:
            t0 = time.perf_counter()
            got[key] = fn()
            dt = time.perf_counter() - t0
            if i >= warmup:
                (ts if key == "s" else tb).append(dt)
        identical &= same(got["s"], got["b"])
        if first is None:
            first = int(got["s"][0])
    us = lambda t: dict(median=1e6 * float(np.median(t)), p90=1e6 * float(np.percentile(t, 90)))  # noqa: E731
    return dict(single_us=us(ts), batch_us=us(tb), identical=bool(identical), nmatches=first)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--label", default="")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--calls", type=int, default=300)
    a = ap.parse_args()
    rng = np.random.default_rng(1)
    euroc = frames(752, 480, 1000, 20220406)
    kitti = frames(1241, 376, 4000, 20220405)
    res = {id(f): ResidentFrame().upload(f) for f in euroc + kitti}
    m_proj, m_init, m_bow = ORBmatcher(0.9, True), ORBmatcher(0.9, True), ORBmatcher(0.75, True)
    rows = []
    for operands in ("host", "resident"):
        op = (lambda f: f) if operands == "host" else (lambda f: res[id(f)])
        shapes = [
            ("match_window 1000 -> 752x480", euroc, window_pair(m_proj, euroc[0], euroc[1], op(euroc[1]))),
            ("match_window 4000 -> 1241x376", kitti, window_pair(m_proj, kitti[0], kitti[1], op(kitti[1]))),
            ("SearchForInitialization 1241x376 / 4000, window 100", kitti, init_pair(m_init, kitti[0], op(kitti[0]),
                                                                                      op(kitti[1]))),
            ("SearchByBoW mode 0, 752x480", euroc, bow_pair(m_bow, euroc[0], euroc[1], op(euroc[0]), op(euroc[1]), 0,
                                                           rng)),
            ("SearchByBoW mode 1, 752x480", euroc, bow_pair(m_bow, euroc[0], euroc[1], op(euroc[0]), op(euroc[1]), 1,
                                                           rng)),
        ]
        for name, fr, (single, batch) in shapes:
            r = dict(shape=name, operands=operands, n1=int(fr[0].N), n2=int(fr[1].N))
            r.update(measure(single, batch, a.warmup, a.calls))
            rows.append(r)
            print(f"{name:55s} {operands:9s} single {r['single_us']['median']:8.1f} us (p90 {r['single_us']['p90']:8.1f})"
                  f"  one-job batch {r['batch_us']['median']:8.1f} us (p90 {r['batch_us']['p90']:8.1f})"
                  f"  identical {r['identical']}  nmatches {r['nmatches']}", flush=True)
    name, power = card()
    out = dict(tool="tools/single_call_probe.py", label=a.label, card=name, power_limit=power, warmup=a.warmup,
               calls=a.calls, timer="host perf_counter around each call (each call ends in a stream synchronise), "
                                    "single and one-job batch alternated call by call, first of the pair alternated",
               shapes=rows)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    return 0 if all(r["identical"] for r in rows) else 1


if __name__ == "__main__":
    sys.exit(main())
