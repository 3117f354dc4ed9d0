"""bench.py --dump-outputs: the file holds what the headline path computed in its last timed step, i.e. the filtered cloud
of frame warmup + steps - 1 of the bench sequence (C2, seed 2), bit for bit the oracle's."""
import subprocess
import sys

import numpy as np
import pytest

from dynamicslamtool_b200 import MovingObjectRemoval, Synth
from helpers import ROOT

pytestmark = pytest.mark.gpu


def test_bench_dumps_the_last_timed_frame(oracle, built, tmp_path):
    steps, warmup = 4, 3
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--no-cpu",
                          "--sequences", "1", "--e2e-sequences", "1", "--c5-sequences", "0", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    got = np.load(out / "filtered_cloud.npy")
    orc = MovingObjectRemoval(ROOT / "config" / "MOR_config_hdl64.txt", 4, 3, binding=oracle)
    s = Synth(2, 2)
    for f in range(warmup + steps):
        orc.push_raw_cloud_and_pose(*s.frame(f))
        want = orc.filter_cloud()
    assert got.dtype == np.float32 and got.shape == want.shape and want.shape[0] > 0
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
