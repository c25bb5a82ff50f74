"""Builds and runs tests/mappoints_wrapper_test.cpp: the C++ drop-ins ORB_SLAM2::MapPointTable and the MapPointTable
overloads of ORBmatcher::SearchByProjection on Frame / MapPoint doubles, against the reference's host path
(Tracking::SearchLocalPoints with isInFrustum on the CPU, and the host-array SearchByProjection calls)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp):
    exe = os.path.join(tmp, "mappoints_wrapper_test")
    lib_dir = os.path.join(ROOT, "swarmmap_b200")
    # -ffp-contract=off: the host-path isInFrustum double must round each product and sum as the reference does
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-o", exe,
                    os.path.join(ROOT, "tests", "mappoints_wrapper_test.cpp"), "-L", lib_dir, "-lswm_orb",
                    "-Wl,-rpath," + lib_dir], check=True)
    return exe


def test_mappoints_wrapper_compiles_and_links(swm, tmp_path):
    assert os.path.exists(_build(str(tmp_path)))


@pytest.mark.gpu
def test_mappoints_wrapper_run(swm, tmp_path):
    exe = _build(str(tmp_path))
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "MAPPOINTS_WRAPPER_OK" in r.stdout, r.stdout + r.stderr
