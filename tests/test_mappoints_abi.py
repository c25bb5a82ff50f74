"""The MapPoint table and the tracking projections (swm_mappoints_*, swm_match_local_map*, swm_match_last_frame): without
a GPU they refuse to run (no CPU fallback); argument checks happen before any device work."""
import ctypes as C

import numpy as np
import pytest


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_no_cpu_fallback(swm):
    if _has_gpu():
        pytest.skip("GPU present: the loud-failure path is exercised on the CPU-only box")
    lib = swm.load()
    t = C.c_void_p()
    assert lib.swm_mappoints_create(0, 100, C.byref(t)) == -3 and not t.value
    assert b"no CPU fallback" in lib.swm_mappoints_last_error(None)
    from swarmmap_b200.matcher import MapPointTable
    with pytest.raises(swm.SwmError):
        MapPointTable()


def test_bad_arguments_rejected_before_device_work(swm):
    lib = swm.load()
    t = C.c_void_p()
    assert lib.swm_mappoints_create(0, -1, C.byref(t)) == -1
    assert lib.swm_mappoints_create(0, 10, None) == -1
    rows = np.zeros(1, np.int32)
    assert lib.swm_mappoints_upsert(None, 1, swm.ptr(rows), None, None, None, None, None, None, None) == -1
    assert lib.swm_mappoints_size(None) == 0
    assert lib.swm_match_local_map_batch(None, None, 0) == -1
    n = C.c_int(0)
    assert lib.swm_match_local_map(None, None, None, None, None, 0, None, 1.0, 0.8, None, None, C.byref(n), None) == -1
    assert lib.swm_match_last_frame(None, None, None, None, None, None, None, 15.0, 1, None, C.byref(n)) == -1
    thr = np.zeros(7, np.float32)
    assert lib.swm_predict_scale_thresholds(0.18232156, 8, swm.ptr(thr)) == 0  # host only: no device needed
    assert (np.diff(thr) > 0).all()


def test_struct_layouts_match_the_header(swm):
    """swm_projection and swm_localmap_job as a C compiler lays them out (the ctypes mirrors in _lib.py)."""
    import os
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "swm_orb.h"\n'
           'int main(void){printf("%zu %zu %zu %zu %zu\\n", sizeof(swm_projection), sizeof(swm_localmap_job),'
           ' offsetof(swm_localmap_job, track), offsetof(swm_localmap_job, n_to_match), sizeof(swm_track_out));}\n')
    with tempfile.TemporaryDirectory() as d:
        c, exe = os.path.join(d, "l.c"), os.path.join(d, "l")
        open(c, "w").write(src)
        subprocess.run(["gcc", "-I", os.path.join(root, "include"), c, "-o", exe], check=True)
        got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    J = swm.LocalMapJob
    assert got == [C.sizeof(swm.Projection), C.sizeof(J), J.track.offset, J.n_to_match.offset, C.sizeof(swm.TrackOut)]
