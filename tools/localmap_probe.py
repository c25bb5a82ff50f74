"""SearchLocalPoints for many agents per call: the resident MapPoint table (swm_match_local_map_batch: row indices and
poses up, projection on the device) against host projection plus swm_match_window_batch (the projected window query of
every point up), on the same synthetic local maps.  Prints one JSON line: device ms, host wall ms and bytes uploaded per
step for both paths, the parity of their results, and the card's name and power limit read in the same run.

  python tools/localmap_probe.py [--agents 128] [--steps 10] [--points 2000]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import frustum_cases as FC  # noqa: E402
import frustum_ref  # noqa: E402
from swarmmap_b200 import _lib  # noqa: E402
from swarmmap_b200.matcher import ORBmatcher  # noqa: E402
from localmap_scenes import make_world, points_kw, resident, upload_table  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--agents", type=int, default=128)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--points", type=int, default=2000)
    a = ap.parse_args()
    rng = np.random.default_rng(7)
    P = a.agents
    worlds = [make_world(rng, a.points) for _ in range(P)]
    rfs = [resident(w["F"]) for w in worlds]
    tables = [upload_table(w["tab"]) for w in worlds]
    m = ORBmatcher(0.8, True)
    lib = _lib.load()
    jobs = [points_kw(w, rf, t, 1.0) for w, rf, t in zip(worlds, rfs, tables)]

    def host_path():
        t0 = time.perf_counter()
        win = []
        for w, rf in zip(worlds, rfs):
            tr, q, blocked, _ = frustum_ref.local_map_query(w["tab"], w["rows"], w["frame_rows"], w["T"], w["K"], w["b4"],
                                                            FC.SF, FC.LOG_SF, 8, 1.0)
            win.append(dict(tgt=rf, desc=q["desc"], u=q["u"], v=q["v"], radius=q["radius"], min_level=q["min_level"],
                            max_level=q["max_level"], valid=q["valid"], blocks=q["blocks"], th_dist=100, ratio_mode=1,
                            tgt_blocked=blocked, check_ori=False))
        t1 = time.perf_counter()
        r = m.match_window_batch(win)
        t2 = time.perf_counter()
        return r, t1 - t0, t2 - t1, lib.swm_matcher_last_device_ms(m._h)

    def table_path():
        t0 = time.perf_counter()
        r = m.search_local_map_batch(jobs)
        return r, time.perf_counter() - t0, lib.swm_matcher_last_device_ms(m._h)

    for _ in range(2):  # warm-up of both shapes
        host_path()
        table_path()
    hp, hc, hd, tw, td = [], [], [], [], []
    parity = True
    for _ in range(a.steps):  # alternate the two paths inside one run
        rh, proj_s, call_s, dev_ms = host_path()
        rt, wall_s, tdev = table_path()
        hp.append(proj_s); hc.append(call_s); hd.append(dev_ms); tw.append(wall_s); td.append(tdev)
        parity &= all(x[0] == y[0] and np.array_equal(x[1], y[1]) for x, y in zip(rh, rt))
    M = sum(len(w["rows"]) for w in worlds)
    N2 = sum(w["F"].N for w in worlds)
    name, power = card()
    print(json.dumps(dict(
        agents=P, steps=a.steps, points_per_agent=a.points, card=name, power_limit=power, parity=bool(parity),
        table_device_ms=float(np.median(td)), table_host_wall_ms=1e3 * float(np.median(tw)),
        table_upload_bytes_computed=4 * M + 8 * N2 + P * 768,  # rows, frame rows, assignments, job records
        host_device_ms=float(np.median(hd)), host_projection_ms=1e3 * float(np.median(hp)),
        host_call_wall_ms=1e3 * float(np.median(hc)), host_upload_bytes_computed=58 * M + 5 * N2 + P * 256,
        note=("upload bytes are computed from the shapes, not counted; the host path's projection is the numpy reading "
              "(tests/frustum_ref.py), not the C++ wrapper's loop, so host wall times of the two C++ paths are not "
              "compared here"))))
    return 0 if parity else 1


if __name__ == "__main__":
    sys.exit(main())
