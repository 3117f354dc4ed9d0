"""Cluster taps of the crop ground mode (k_frame and k_frame_pipe) against the oracle on C2, dense frames included: the
clusters' centroids and boxes are summed per cell and per component before the select, and a pipelined launch writes
the per-point labels and cluster ids in the back half of the frame, from buffers the next frame's front half does not
touch. Labels, cluster ids, centroids and boxes (and every other tap) must still equal the oracle's, with one kernel per
frame and with pipelined launches."""
import ctypes as C

import numpy as np
import pytest

from dynamicslamtool_b200 import MovingObjectRemoval, Synth
from parity import ParityStats, compare_frame

pytestmark = pytest.mark.gpu

FRAMES = range(98, 108)  # C2 including its dense frames 101-107 (a mover at 1.7 m: cells with > 1000 points)
CHECKPOINTS = {0, 1, 2, 4, 6, 8, 9}  # (the frames in between leave their back half to the next frame's fused launch)


@pytest.mark.parametrize("pipelining", [False, True])
def test_c2_cluster_taps_equal_oracle(product, oracle, cfg_dir, pipelining):
    cfg = cfg_dir / "MOR_config_hdl64.txt"
    s = Synth(2, 2)
    seq = [s.frame(f) for f in FRAMES]
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=s.max_points)
    gpu.set_pipelining(pipelining)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    d = []
    try:
        for pts, _ in seq:
            p = C.c_void_p()
            assert product.device_alloc(0, max(pts.nbytes, 16), C.byref(p)) == 0
            assert product.device_upload(0, p, pts.ctypes.data_as(C.c_void_p), pts.nbytes) == 0
            d.append(p)
        stats = ParityStats()
        for f, (pts, pose) in enumerate(seq):
            gpu.push_device(d[f].value, len(pts), pose)
            gpu.filter_device(None, 0, want_count=False)
            orc.push_raw_cloud_and_pose(pts, pose)
            oo = orc.filter_cloud().copy()
            if f not in CHECKPOINTS:
                continue
            n = gpu.counts()["NOUT"]
            og = np.empty((n, 8), np.float32)
            if n:
                assert product.device_download(0, og.ctypes.data_as(C.c_void_p), C.c_void_p(gpu.output_device()), og.nbytes) == 0
            bad = compare_frame(gpu, orc, og, oo, stats)
            assert not bad, f"frame {FRAMES[f]}: {bad}"
        assert stats.matches > 0 and stats.frames == len(CHECKPOINTS)
    finally:
        for p in d:
            product.device_free(0, p)
        gpu.close()
