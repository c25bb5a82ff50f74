"""Builds and runs tests/kfdb_wrapper_test.cpp: the C++ drop-ins ORB_SLAM2::KeyFrameDatabase and ORBVocabulary::score
on KeyFrame / Frame doubles, with the reference's call sites, against the KeyFrameDatabase oracle."""
import os
import subprocess

import pytest

import oracle_kfdb_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp):
    exe = os.path.join(tmp, "kfdb_wrapper_test")
    oracle_kfdb_lib.build()
    lib_dirs = [os.path.join(ROOT, "swarmmap_b200"), os.path.join(ROOT, "oracle")]
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(ROOT, "tests", "kfdb_wrapper_test.cpp"),
                    "-L", lib_dirs[0], "-lswm_orb", "-L", lib_dirs[1], "-l:liborb_oracle_kfdb.so"] +
                   ["-Wl,-rpath," + d for d in lib_dirs], check=True)
    return exe


def test_kfdb_wrapper_compiles_and_links(swm, tmp_path):
    assert os.path.exists(_build(str(tmp_path)))


@pytest.mark.gpu
def test_kfdb_wrapper_run(swm, tmp_path):
    exe = _build(str(tmp_path))
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "KFDB_WRAPPER_OK" in r.stdout, r.stdout + r.stderr
