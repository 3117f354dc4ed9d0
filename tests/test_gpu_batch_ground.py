"""mor_batch_step_device with the voxel-covariance ground modes (ground_mode 1 and 2, -m gpu).

Every sequence of a batch is checked against the CPU oracle with the checks of test_voxel_covariance_ground_modes (voxel
count, accepted flags and bins exact, centroids and normals within 1e-5, compare_frame downstream) and, where a test
says so, byte for byte against an unbatched GPU handle ("twin") that is fed the same frames through push_device +
filter_device."""
import ctypes as C

import numpy as np
import pytest

from dynamicslamtool_b200 import MovingObjectRemoval, SequenceBatch, Synth
from helpers import write_cfg
from parity import compare_frame

pytestmark = pytest.mark.gpu

C4_CELLS = 1 << 21  # C4 at leaf 0.5 spans ~1.2e5 voxels: 37 handles of this size fit easily beside other work
TWIN_TAPS = ("labels", "cluster_id", "flags", "removed_mask")


def _alloc(product, nbytes):
    p = C.c_void_p()
    assert product.device_alloc(0, nbytes, C.byref(p)) == 0
    return p


class Bed:
    """S batched handles (optionally with unbatched twins) and their device input / output buffers."""

    def __init__(self, product, cfg, S, maxp, max_cells=C4_CELLS, twins=False):
        self.p, self.maxp = product, maxp
        make = lambda: MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=maxp, max_cells=max_cells)  # noqa: E731
        self.gpus = [make() for _ in range(S)]
        self.twins = [make() for _ in range(S)] if twins else []
        self.batch = SequenceBatch(self.gpus)
        self.d_in = [_alloc(product, maxp * 32) for _ in range(S)]
        self.d_out = [_alloc(product, maxp * 32) for _ in range(S)]
        self.d_tout = [_alloc(product, maxp * 32) for _ in self.twins]

    def step(self, recs, ns, poses, point_step=16, offsets=(0, 4, 8, 12)):
        """recs[s]: the records of sequence s (any dtype, C-contiguous), ns[s] points."""
        for h in self.gpus + self.twins:  # the uploads below overwrite what the last step read
            h.sync()
        for s, r in enumerate(recs):
            if r.nbytes:
                assert self.p.device_upload(0, self.d_in[s], r.ctypes.data_as(C.c_void_p), r.nbytes) == 0
        self.batch.step_device([p.value for p in self.d_in], ns, poses, [p.value for p in self.d_out], point_step, offsets)
        for s, t in enumerate(self.twins):
            t.push_device(self.d_in[s].value, ns[s], poses[s], point_step, offsets)
            t.filter_device(self.d_tout[s].value, self.maxp, want_count=False)

    def _download(self, h, d):
        h.sync()
        n = h.counts()["NOUT"]
        out = np.empty((n, 8), np.float32)
        if n:
            assert self.p.device_download(0, out.ctypes.data_as(C.c_void_p), d, n * 32) == 0
        return out

    def output(self, s):
        return self._download(self.gpus[s], self.d_out[s])

    def twin_output(self, s):
        return self._download(self.twins[s], self.d_tout[s])

    def assert_twin(self, s, where):
        g, t = self.gpus[s], self.twins[s]
        assert g.counts() == t.counts(), f"{where}: counts {g.counts()} vs unbatched {t.counts()}"
        assert self.output(s).tobytes() == self.twin_output(s).tobytes(), f"{where}: output records differ from the unbatched handle"
        for tap in TWIN_TAPS:
            assert g.tap(tap).tobytes() == t.tap(tap).tobytes(), f"{where}: {tap} differs from the unbatched handle"

    def close(self):
        for p in self.d_in + self.d_out + self.d_tout:
            self.p.device_free(0, p)


@pytest.fixture
def beds():
    made = []
    yield made
    for b in made:
        b.close()


def oracle_step(orc, recs, pose, **kw):
    """push + filter on the oracle; returns (ground voxels after the push, output records)."""
    orc.push_raw_cloud_and_pose(recs, pose, **kw)
    vo = orc.tap("ground_voxels")
    return vo, orc.filter_cloud().copy()


def assert_oracle(gpu, orc, out, vo, oo, where):
    """The checks of test_voxel_covariance_ground_modes for one batched sequence."""
    vg = gpu.tap("ground_voxels")
    assert vg.shape == vo.shape and vg.shape[0] > 0, f"{where}: voxel count {vg.shape} vs {vo.shape}"
    np.testing.assert_allclose(vg[:, :3], vo[:, :3], rtol=1e-5, atol=1e-7, err_msg=f"{where}: voxel centroids")
    assert np.array_equal(vg[:, 3], vo[:, 3]), f"{where}: accepted flags differ in {int(np.sum(vg[:, 3] != vo[:, 3]))} voxels"
    acc = vo[:, 3] > 0
    assert np.array_equal(vg[acc, 4], vo[acc, 4]), f"{where}: bin keys"
    np.testing.assert_allclose(vg[acc, 5:], vo[acc, 5:], rtol=1e-5, atol=1e-6, err_msg=f"{where}: normals")
    bad = compare_frame(gpu, orc, out, oo)
    assert not bad, f"{where}: {bad}"


def oracles(oracle, cfg, n):
    return [MovingObjectRemoval(cfg, 4, 3, binding=oracle) for _ in range(n)]


@pytest.mark.parametrize("scenario,base,overrides", [
    (4, "MOR_config_terrain.txt", {}),                                 # C4: eigen-normal mode on sloped / multi-plane terrain
    (4, "MOR_config_terrain.txt", {"ground_mode": 1, "gp_leaf": 0.5}),
    (1, "MOR_config.txt", {"ground_mode": 1}),                         # literal mode with the reference defaults (leaf 0.1)
    (1, "MOR_config.txt", {"ground_mode": 2, "gp_bin_width": 0.1}),
])
def test_batched_ground_modes_match_oracle_and_unbatched(product, oracle, cfg_dir, tmp_path, beds, scenario, base, overrides):
    S, frames = 3, 8
    cfg = write_cfg(tmp_path, base=cfg_dir / base, **overrides)
    syn = [Synth(scenario, 40 + s) for s in range(S)]
    bed = Bed(product, cfg, S, syn[0].max_points, twins=True)
    beds.append(bed)
    orcs = oracles(oracle, cfg, S)
    for f in range(frames):
        data = [syn[s].frame(f) for s in range(S)]
        bed.step([d[0] for d in data], [d[0].shape[0] for d in data], [d[1] for d in data])
        for s in range(S):
            vo, oo = oracle_step(orcs[s], *data[s])
            assert_oracle(bed.gpus[s], orcs[s], bed.output(s), vo, oo, f"sequence {s} frame {f}")
            assert bed.gpus[s].counts()["NG"] > 0
            bed.assert_twin(s, f"sequence {s} frame {f}")


def test_batched_ground_at_the_benchmarked_width(product, oracle, cfg_dir, beds):
    """37 sequences per launch on C4 (mode 2): 8 distinct streams, each repeated inside the batch. The copies agree bit
    for bit, and every stream matches the oracle."""
    S, frames = 37, 6
    cfg = cfg_dir / "MOR_config_terrain.txt"
    streams = [(4, 0), (4, 10), (5, 0), (6, 3), (7, 0), (8, 5), (9, 0), (10, 2)]
    syn = [Synth(4, seed) for seed, _ in streams]
    bed = Bed(product, cfg, S, syn[0].max_points)
    beds.append(bed)
    orcs = oracles(oracle, cfg, len(streams))
    for f in range(frames):
        data = [syn[t].frame(streams[t][1] + f) for t in range(len(streams))]
        bed.step([data[s % 8][0] for s in range(S)], [data[s % 8][0].shape[0] for s in range(S)], [data[s % 8][1] for s in range(S)])
        outs = [bed.output(s) for s in range(S)]
        for t in range(len(streams)):
            vo, oo = oracle_step(orcs[t], *data[t])
            assert_oracle(bed.gpus[t], orcs[t], outs[t], vo, oo, f"stream {t} frame {f}")
            for c in range(t + 8, S, 8):
                assert outs[t].tobytes() == outs[c].tobytes(), f"copy {c} of stream {t} differs at frame {f}"
                assert bed.gpus[t].counts() == bed.gpus[c].counts(), f"counts: copy {c} of stream {t} at frame {f}"
                for tap in ("labels", "cluster_id", "centroids", "flags", "mo_conf", "removed_mask", "ground_voxels"):
                    assert bed.gpus[t].tap(tap).tobytes() == bed.gpus[c].tap(tap).tobytes(), f"{tap}: copy {c} of stream {t} differs at frame {f}"


def test_unequal_frames_in_one_batch(product, cfg_dir, beds):
    """Frames of very different sizes in one step (an empty one, a few hundred points, full C4 frames; the leader small
    too): the point-indexed stages are sized for the largest, and every sequence equals its unbatched twin."""
    S = 4
    cfg = cfg_dir / "MOR_config_terrain.txt"
    syn = [Synth(4, 60 + s) for s in range(S)]
    bed = Bed(product, cfg, S, syn[0].max_points, twins=True)
    beds.append(bed)
    # per frame: points each sequence gets (None = the whole frame)
    plan = [[None] * 4, [None] * 4, [None, 0, 300, None], [0, None, None, 300], [None, 300, 0, None], [None] * 4]
    for f, sizes in enumerate(plan):
        data = [syn[s].frame(f) for s in range(S)]
        recs = [np.ascontiguousarray(d[0][: (len(d[0]) if k is None else k)]) for d, k in zip(data, sizes)]
        bed.step(recs, [r.shape[0] for r in recs], [d[1] for d in data])
        for s in range(S):
            bed.assert_twin(s, f"sequence {s} frame {f} ({recs[s].shape[0]} points)")


def test_ground_capacity_error_stays_in_its_sequence(product, oracle, cfg_dir, beds):
    """A frame whose bounding box needs more than max_cells cells (one point at z = 1e3) raises ERR_GROUND_CAP (8) in its
    own sequence's counts, as an unbatched handle does for the same frame; the other sequences match the oracle."""
    S, bad_seq, bad_frame = 3, 1, 2
    cfg = cfg_dir / "MOR_config_terrain.txt"
    syn = [Synth(4, 70 + s) for s in range(S)]
    maxp = syn[0].max_points + 1
    bed = Bed(product, cfg, S, maxp, max_cells=1 << 20, twins=True)
    beds.append(bed)
    orcs = oracles(oracle, cfg, S)
    for f in range(4):
        data = [syn[s].frame(f) for s in range(S)]
        recs = [d[0] for d in data]
        if f == bad_frame:
            recs[bad_seq] = np.ascontiguousarray(np.concatenate([recs[bad_seq], np.float32([[1.0, 1.0, 1e3, 0.5]])]))
        bed.step(recs, [r.shape[0] for r in recs], [d[1] for d in data])
        for s in range(S):
            where = f"sequence {s} frame {f}"
            err = bed.gpus[s].counts()["ERRFLAGS"]
            if s == bad_seq and f >= bad_frame:
                if f == bad_frame:
                    assert err & 8, f"{where}: ERRFLAGS {err}"
                bed.assert_twin(s, where)  # same error bits, same results as the unbatched handle
                continue
            assert err == 0, f"{where}: ERRFLAGS {err}"
            vo, oo = oracle_step(orcs[s], recs[s], data[s][1])
            assert_oracle(bed.gpus[s], orcs[s], bed.output(s), vo, oo, where)


@pytest.mark.parametrize("S", [1, 3, 37])
def test_launch_count_per_ground_step(product, cfg_dir, beds, S):
    """9 ground launches + 1 frame launch per batched step on the leader, whatever S; the followers launch nothing."""
    cfg = cfg_dir / "MOR_config_terrain.txt"
    syn = Synth(4, 80)
    bed = Bed(product, cfg, S, syn.max_points)
    beds.append(bed)
    for f in range(3):
        pts, pose = syn.frame(f)
        before = [g.launch_count() for g in bed.gpus]
        bed.step([pts] * S, [pts.shape[0]] * S, [pose] * S)
        after = [g.launch_count() for g in bed.gpus]
        assert after[0] - before[0] == 10, (f, before[0], after[0])
        assert after[1:] == before[1:]


@pytest.mark.parametrize("case", ["xyzirt22", "method1"])
def test_batched_ground_layouts_and_method_1(product, oracle, cfg_dir, tmp_path, beds, case):
    """22-byte XYZIRT records (the byte-assembled read of the ground ingest) and the point-distance moving test
    (method_choice 1) with ground mode 2: every sequence matches the oracle."""
    S, frames = 3, 5
    base = cfg_dir / "MOR_config_terrain.txt"
    cfg = write_cfg(tmp_path, base=base, method_choice=1) if case == "method1" else base
    syn = [Synth(4, 90 + s) for s in range(S)]
    bed = Bed(product, cfg, S, syn[0].max_points)
    beds.append(bed)
    orcs = oracles(oracle, cfg, S)
    step_b, offs = (22, (0, 4, 8, 12)) if case == "xyzirt22" else (16, (0, 4, 8, 12))
    for f in range(frames):
        data = [syn[s].frame(f) for s in range(S)]
        recs = []
        for pts, _ in data:
            if case == "xyzirt22":
                rec = np.full((len(pts), 22), 0xA5, np.uint8)
                for col, off in enumerate(offs):
                    rec[:, off:off + 4] = pts[:, col:col + 1].copy().view(np.uint8)
                recs.append(np.ascontiguousarray(rec))
            else:
                recs.append(pts)
        bed.step(recs, [d[0].shape[0] for d in data], [d[1] for d in data], point_step=step_b, offsets=offs)
        for s in range(S):
            kw = dict(point_step=step_b, offsets=offs) if case == "xyzirt22" else {}
            vo, oo = oracle_step(orcs[s], recs[s], data[s][1], **kw)
            assert_oracle(bed.gpus[s], orcs[s], bed.output(s), vo, oo, f"{case} sequence {s} frame {f}")


def test_ground_batch_and_single_stepping_alternate(product, oracle, cfg_dir, beds):
    """The leader and a follower leave the batch for single stepping and rejoin it; parity with the oracle holds
    throughout (the crop-mode counterpart is test_batched_step_matches_oracle_per_sequence)."""
    S = 3
    cfg = cfg_dir / "MOR_config_terrain.txt"
    syn = [Synth(4, 100 + s) for s in range(S)]
    bed = Bed(product, cfg, S, syn[0].max_points)
    beds.append(bed)
    orcs = oracles(oracle, cfg, S)

    def batched(f):
        data = [syn[s].frame(f) for s in range(S)]
        bed.step([d[0] for d in data], [d[0].shape[0] for d in data], [d[1] for d in data])
        for s in range(S):
            vo, oo = oracle_step(orcs[s], *data[s])
            assert_oracle(bed.gpus[s], orcs[s], bed.output(s), vo, oo, f"batched sequence {s} frame {f}")

    def single(f):
        for s in range(S):
            pts, pose = syn[s].frame(f)
            g = bed.gpus[s]
            g.push_raw_cloud_and_pose(pts, pose)
            vg = g.tap("ground_voxels").copy()
            og = g.filter_cloud().copy()
            vo, oo = oracle_step(orcs[s], pts, pose)
            assert vg.shape == vo.shape and np.array_equal(vg[:, 3], vo[:, 3]), f"single sequence {s} frame {f}: ground voxels"
            bad = compare_frame(g, orcs[s], og, oo)
            assert not bad, f"single sequence {s} frame {f}: {bad}"

    for f in range(3):
        batched(f)
    single(3)
    single(4)
    for f in range(5, 7):
        batched(f)
    single(7)
    batched(8)
