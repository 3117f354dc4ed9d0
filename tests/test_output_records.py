"""The expected filtered cloud in record layout (tests/records_ref.py), checked on the CPU oracle alone: the source indices
derived from the oracle's point-class and removal-mask taps reproduce its PointXYZI output point for point, for every
record layout the GPU tests use. The GPU's record output is held to this derivation in test_gpu_output_records.py."""
import numpy as np
import pytest

from dynamicslamtool_b200 import MovingObjectRemoval, Synth
from dynamicslamtool_b200.binding import NO_FIELD
from helpers import IDENTITY_POSE, OPEN_CFG, blob, with_intensity, write_cfg
from records_ref import LAYOUTS, PAD, expected_records, expected_sources, fields_of, make_records


def _check_frame(orc, rec, offs, where):
    xyzi = orc.filter_cloud().copy()
    src = expected_sources(orc)
    assert len(src) == len(xyzi), f"{where}: {len(src)} sources for {len(xyzi)} output points"
    pc, rm = orc.tap("point_class"), orc.tap("removed_mask")
    nk = int(np.sum((pc == 1) & (rm != 2)))
    kept, ground = src[:nk], src[nk:]
    assert np.all(np.diff(kept) > 0) and np.all(np.diff(ground) > 0), f"{where}: sources not ascending"
    assert np.all(rm[kept] == 1) and np.all(pc[ground] == 2)
    got = expected_records(orc, rec)
    assert got.shape == (len(xyzi), rec.shape[1])
    f = fields_of(got, offs)
    # the x/y/z/intensity fields of the records are the PointXYZI output, bit for bit, in order
    assert f[:, :3].tobytes() == np.ascontiguousarray(xyzi[:, :3]).tobytes(), f"{where}: xyz differ"
    want_i = xyzi[:, 4] if offs[3] != NO_FIELD else np.zeros(len(xyzi), np.float32)
    assert f[:, 3].tobytes() == np.ascontiguousarray(want_i).tobytes(), f"{where}: intensity differs"
    return got


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_records_from_oracle_on_c1(oracle, cfg_dir, layout):
    s = Synth(1, 1)
    orc = MovingObjectRemoval(cfg_dir / "MOR_config.txt", 4, 3, binding=oracle)
    removed = 0
    for f in range(8):
        pts, pose = s.frame(f)
        rec, step, offs = make_records(pts, layout)
        orc.push_raw_cloud_and_pose(rec, pose, point_step=step, offsets=offs)
        got = _check_frame(orc, rec, offs, f"frame {f}")
        removed += int(np.sum(orc.tap("removed_mask") == 2))
        if LAYOUTS[layout][2]:  # ring / time travel with their points
            ring = np.ascontiguousarray(got[:, 16:18]).view("<u2").reshape(-1)
            assert np.array_equal(ring, (expected_sources(orc) % 16).astype(np.uint16))
    assert removed > 0  # the sequence removes moving points: the kept list is not the whole cloud


@pytest.mark.parametrize("seed", range(4))
def test_records_from_oracle_on_random_blob_scenes(oracle, tmp_path, seed):
    rng = np.random.default_rng(300 + seed)
    cfg = write_cfg(tmp_path, ec_distance_threshold=0.3, min_cluster_size=30, max_cluster_size=5000,
                    **{**OPEN_CFG, "gp_limit": -0.5})
    orc = MovingObjectRemoval(cfg, 2, 2, binding=oracle)
    layout = sorted(LAYOUTS)[seed % len(LAYOUTS)]
    centers = rng.uniform(-4, 4, (4, 3)).astype(np.float32)
    speed = rng.uniform(-0.3, 0.3, (4, 3)).astype(np.float32)
    ground = np.concatenate([rng.uniform(-5, 5, (400, 2)), np.full((400, 1), -1.0)], axis=1).astype(np.float32)
    for f in range(6):
        parts = [blob(rng, centers[k] + f * speed[k], int(rng.integers(80, 300)), 0.1) for k in range(4)] + [ground]
        pts = with_intensity(np.concatenate(parts), 0.75)
        pts[:, 3] = rng.uniform(0, 1, len(pts)).astype(np.float32)
        perm = rng.permutation(len(pts))  # cloud and ground points interleaved in input order
        pts = np.ascontiguousarray(pts[perm])
        rec, step, offs = make_records(pts, layout)
        orc.push_raw_cloud_and_pose(rec, IDENTITY_POSE, point_step=step, offsets=offs)
        _check_frame(orc, rec, offs, f"seed {seed} frame {f}")
        assert orc.counts()["NG"] > 0


def test_make_records_layouts():
    pts = np.arange(12, dtype=np.float32).reshape(3, 4)
    for name, (step, offs, extra) in LAYOUTS.items():
        rec, st, of = make_records(pts, name)
        assert rec.shape == (3, step) and st == step and of == offs
        assert np.array_equal(fields_of(rec, offs)[:, :3], pts[:, :3])
        used = np.zeros(step, bool)
        for off in offs:
            if off != NO_FIELD:
                used[off:off + 4] = True
        for off, dt in extra.values():
            used[off:off + np.dtype(dt).itemsize] = True
        assert np.all(rec[:, ~used] == PAD)
    for name in LAYOUTS:  # an empty frame
        assert make_records(np.zeros((0, 4), np.float32), name)[0].shape == (0, LAYOUTS[name][0])
    rec, _, _ = make_records(np.zeros((40, 4), np.float32), "xyzirt22")
    t = np.ascontiguousarray(rec[:, 18:22]).view("<f4").reshape(-1)
    assert len(np.unique(t)) == 40  # a distinct time per point
