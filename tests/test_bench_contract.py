"""The bench.py JSON contract, checked on the committed lines (profiles/r2am_bench.json from `python bench.py` on one
B200, profiles/r2ae_bench_reference.json from `python bench.py --impl reference`), and the parts of bench.py that run
without a GPU (argument parsing, the reference arm on a tiny sample); on the GPU, what `--dump-outputs` writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV_LINE = "r2am_bench.json"


def _line(name):
    with open(os.path.join(ROOT, "profiles", name)) as f:
        return json.loads(f.read().strip().splitlines()[-1])


def test_device_arm_line_has_every_contract_key():
    d = _line(DEV_LINE)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
        assert k in d, k
    # BASELINE.json's metric is prose ("ORB frames/sec/GPU (1000 feat, 752x480) ...; Hamming matches/sec"): the line
    # carries the first as `value` (whole-job frames/s) and the second under "hamming"
    assert "ORB frames/sec" in base["metric"] and "Hamming matches/sec" in base["metric"]
    assert d["metric"] == "orb_extract_frames_per_sec" and d["unit"] == "frames/s"
    assert d["hamming"]["metric"] == "hamming_matches_per_sec" and d["hamming"]["value"] > 0
    assert d["config"]["frame"] == [752, 480] and d["config"]["nfeatures"] == 1000
    assert d["n_gpus"] == 1 and d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "u8" and d["data"] == "synthetic" and "workload" in d["config"] and "model" not in d["config"]
    frames_per_step = d["config"]["batch_per_gpu"] * d["n_gpus"]
    assert d["value"] > 0 and abs(d["ms_per_step"] * 1e-3 * d["value"] / frames_per_step - 1) < 0.02
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    assert d["gpu_launches"] > 0
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    # the line was computed against the HBM peak measured on the B200 it was taken on: 6454.3 GB/s (DESIGN.md section 7)
    assert r["peak_source"].startswith("measured") and r["peak"] == 6454.3 and r["traffic"] is not None
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    k = d["clocks"]
    assert k["sm_mhz"] > 0 and k["sm_max_mhz"] >= k["sm_mhz"] and not set(k["reasons"]) & {
        "hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    h = d["hamming"]
    assert h["roofline"]["bound"] == "tensor" and 0 < h["roofline"]["frac"] < 1.2
    assert d["config"]["timed_region_s"] >= 1.0 and e["timed_region_s"] >= 1.0
    assert 0 < e["h2d_ceiling"]["e2e_frac_of_ceiling"] <= 1.05
    # one record per remaining BASELINE.json config, each with its own workload, device value, e2e and a parity check
    w = d["workloads"]
    k2 = w["config2_kitti"]
    assert k2["config"]["frame"] == [1241, 376] and k2["extract"]["value"] > 0 and k2["extract"]["e2e"]["value"] > 0
    assert k2["init_matching"]["value"] > 0 and k2["init_matching"]["parity"]["identical"] is True
    t = w["config34_tracking"]
    assert t["parity"]["identical"] is True
    for variant in ("projection_only", "with_bow"):
        v = t["variants"][variant]
        assert v["value"] >= 5000 and v["e2e"]["value"] >= 5000  # north_star's floor per GPU, with bit-exact matches
    p5 = w["config5_place"]
    assert "100 000 keyframes x 256" in p5["config"]["workload"] and p5["parity"]["votes_on_planted_keyframes"] is True
    assert p5["parity"]["oracle_sample"]["identical"] is True and p5["value"] > 1e12
    proto = d["cpu_baseline_protocol"]
    for variant in ("O2", "O1"):
        assert [x["agents"] for x in proto[variant]["extract"]][:2] == [1, 2] and proto[variant]["matchers"]


def test_reference_arm_line():
    d = _line("r2ae_bench_reference.json")
    dev = _line(DEV_LINE)
    assert d["impl"] == "reference" and d["metric"] == dev["metric"] and d["unit"] == dev["unit"]
    assert d["config"]["workload"] == dev["config"]["workload"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1


def test_reference_arm_runs_without_a_gpu():
    """`bench.py --impl reference` is the CPU oracle on the host cores: it must run on a box without a GPU."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["value"] > 0


def _bench_swm(*extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--warmup", "0", "--batch", "512", "--only", "headline",
                        "--no-cpu-baseline", *extra], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_dump_outputs_are_the_extractor_outputs(oracle, swm, tmp_path):
    """`--steps` sets how many steps run (kernel launches counted in the timed loop), and `--dump-outputs` writes the
    headline's last timed step for a seeded 256-frame sample of the batch: float32, at most 64 MB, for sampled frames
    the same keypoints and descriptors as an extractor handle of its own, and for one frame those of the CPU oracle."""
    import bench
    from swarmmap_b200.orb import KP_DTYPE, ORBextractor
    out = tmp_path / "dump"
    one = _bench_swm("--steps", "1")
    two = _bench_swm("--steps", "2", "--dump-outputs", str(out))
    assert one["steps"] == 1 and two["steps"] == 2 and two["gpu_launches"] == 2 * one["gpu_launches"] > 0
    a = {k: np.load(out / f"{k}.npy") for k in ("frames", "n_keypoints", "keypoints", "descriptors")}
    assert all(v.dtype == np.float32 for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64 << 20
    idx, n = a["frames"].astype(np.int64), a["n_keypoints"].astype(np.int64)
    assert len(idx) == len(n) == 256 and np.all(np.diff(idx) > 0) and idx[-1] < 512
    assert len(a["keypoints"]) == len(a["descriptors"]) == n.sum() and n.min() > 500
    off = np.concatenate([[0], np.cumsum(n)])
    frames = bench.headline_frames(512)
    imgs = frames[idx % len(frames)]
    pos = [0, 101, 255]
    kps, desc, cnt = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=3).extract_batch(imgs[pos])
    for j, i in enumerate(pos):
        assert cnt[j] == n[i]
        k = kps[j, :cnt[j]]
        np.testing.assert_array_equal(a["keypoints"][off[i]:off[i + 1]], np.stack([k[f].astype(np.float32) for f in KP_DTYPE.names], 1))
        np.testing.assert_array_equal(a["descriptors"][off[i]:off[i + 1]], desc[j, :cnt[j]].astype(np.float32))
    # independent of the CUDA path: the oracle's extraction of the last sampled frame, with smoke()'s tolerances
    i = 255
    okps, odesc = oracle.Extractor(1000, 1.2, 8, 20, 7)(imgs[i])
    got = a["keypoints"][off[i]:off[i + 1]]
    assert len(got) == len(okps)
    for c, f in enumerate(KP_DTYPE.names):
        if f not in ("angle", "class_id"):
            np.testing.assert_array_equal(got[:, c], okps[f].astype(np.float32), err_msg=f)
    dang = np.abs(got[:, 3] - okps["angle"])
    assert np.deg2rad(np.minimum(dang, 360 - dang).max()) <= 1e-4
    bits = np.unpackbits(a["descriptors"][off[i]:off[i + 1]].astype(np.uint8) ^ odesc)
    assert 1.0 - bits.sum() / float(bits.size) >= 0.999
