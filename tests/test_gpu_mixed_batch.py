"""mor_batch_step_device_mixed (-m gpu): sequences at different frames, with their own configs, limits, record layouts and
output-record settings, in one step.

Every sequence is checked, after every step, against its own unbatched handle ("twin") fed the same frames through
push_device + filter_device: output bytes, counts, the removal mask, cluster ids, mo_vec (MO_CENTROIDS, MO_CONF) and
flags."""
import ctypes as C

import numpy as np
import pytest

from dynamicslamtool_b200 import MixedBatch, MorError, MovingObjectRemoval, Synth
from helpers import IDENTITY_POSE, write_cfg
from test_gpu_many_clusters import MAX_CLUSTERS, N_BAD, N_GOOD, scene_cfg, scene_frames

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_CAPACITY, ERR_GROUND_CAP = 5, 6, 8
C4_CELLS = 1 << 21
TWIN_TAPS = ("removed_mask", "cluster_id", "mo_centroids", "mo_conf", "flags")
CONFIGS = {1: "MOR_config.txt", 2: "MOR_config_hdl64.txt", 3: "MOR_config_os128.txt", 4: "MOR_config_terrain.txt"}
LAYOUTS = {16: (0, 4, 8, 12), 22: (0, 4, 8, 12), 32: (0, 4, 8, 16)}  # 22: velodyne XYZIRT; 32: x, y, z, pad, intensity, ...


def records(pts, step):
    """float32 [n, 4] points as uint8 [n, step] records of the layout LAYOUTS[step]; the other bytes are a pattern that
    differs from record to record, so a copied record shows where it came from."""
    if step == 16:
        return np.ascontiguousarray(pts, np.float32)
    n = len(pts)
    rec = ((np.arange(n, dtype=np.int64)[:, None] * 7 + np.arange(step)[None, :]) & 0xFF).astype(np.uint8)
    for col, off in enumerate(LAYOUTS[step]):
        rec[:, off:off + 4] = pts[:, col:col + 1].copy().view(np.uint8)
    return np.ascontiguousarray(rec)


class Seq:
    """A batched handle and its unbatched twin, built alike; their device output buffers."""

    def __init__(self, product, cfg, maxp, step=16, out_records=False, n_bad=4, n_good=3, **limits):
        self.p, self.maxp, self.step = product, maxp, step
        make = lambda: MovingObjectRemoval(cfg, n_bad, n_good, binding=product, max_points=maxp, **limits)  # noqa: E731
        self.gpu, self.twin = make(), make()
        for h in (self.gpu, self.twin):
            h.set_output_records(out_records)
        self.rec_bytes = step if out_records else 32
        self.d_out, self.d_tout = _alloc(product, maxp * 32), _alloc(product, maxp * 32)

    def reset(self):
        self.gpu.reset()
        self.twin.reset()

    def _download(self, h, d):
        h.sync()
        n = h.counts()["NOUT"]
        out = np.empty(n * self.rec_bytes, np.uint8)
        if n:
            assert self.p.device_download(0, out.ctypes.data_as(C.c_void_p), d, out.nbytes) == 0
        return out

    def assert_twin(self, where):
        g, t = self.gpu, self.twin
        assert g.counts() == t.counts(), f"{where}: counts {g.counts()} vs unbatched {t.counts()}"
        assert self._download(g, self.d_out).tobytes() == self._download(t, self.d_tout).tobytes(), f"{where}: output bytes differ"
        for tap in TWIN_TAPS:
            assert g.tap(tap).tobytes() == t.tap(tap).tobytes(), f"{where}: {tap} differs from the unbatched handle"


def _alloc(product, nbytes):
    p = C.c_void_p()
    assert product.device_alloc(0, max(nbytes, 16), C.byref(p)) == 0
    return p


class Bed:
    """Device copies of every frame used (uploaded once) and the step / compare loop."""

    def __init__(self, product):
        self.p, self.mixed, self.bufs = product, MixedBatch(product), []

    def upload(self, rec):
        d = _alloc(self.p, rec.nbytes)
        if rec.nbytes:
            assert self.p.device_upload(0, d, rec.ctypes.data_as(C.c_void_p), rec.nbytes) == 0
        self.bufs.append(d)
        return d

    def step(self, seqs, frames, twins=True):
        """frames[s] = (float32 [n, 4] points, pose7): one mixed step, then the same frame on every twin."""
        recs = [records(pts, q.step) for q, (pts, _) in zip(seqs, frames)]
        d_in = [self.upload(r) for r in recs]
        ns = [len(pts) for pts, _ in frames]
        self.mixed.step([q.gpu for q in seqs], [d.value for d in d_in], ns, [pose for _, pose in frames], [q.d_out.value for q in seqs],
                        [q.step for q in seqs], [LAYOUTS[q.step] for q in seqs])
        if twins:
            for q, d, n, (_, pose) in zip(seqs, d_in, ns, frames):
                q.twin.push_device(d.value, n, pose, q.step, LAYOUTS[q.step])
                q.twin.filter_device(q.d_tout.value, q.maxp, want_count=False)

    def check(self, seqs, where):
        for s, q in enumerate(seqs):
            q.assert_twin(f"{where}, sequence {s}")

    def close(self, seqs=()):
        for q in seqs:
            q.gpu.sync()
            q.twin.sync()
        for d in self.bufs:
            self.p.device_free(0, d)
        for q in seqs:
            self.p.device_free(0, q.d_out)
            self.p.device_free(0, q.d_tout)


@pytest.fixture
def bed(product):
    made = {"bed": Bed(product), "seqs": []}
    yield made
    made["bed"].close(made["seqs"])


MAX_POINTS = {}


def synth_seq(product, cfg_dir, scenario, cfg=None, **kw):
    """A Seq with the config and max_points of scenario C<scenario>, or the config `cfg`."""
    if scenario not in MAX_POINTS:
        MAX_POINTS[scenario] = Synth(scenario, 0).max_points
    return Seq(product, cfg or cfg_dir / CONFIGS[scenario], MAX_POINTS[scenario], **kw)


def test_c1_c2_c3_in_one_batch(product, cfg_dir, bed):
    """Three sensors, three configs, three sets of limits in one step, over twelve steps."""
    b, seqs = bed["bed"], bed["seqs"]
    syn = [Synth(sc, 10 + sc) for sc in (1, 2, 3)]
    seqs += [synth_seq(product, cfg_dir, sc) for sc in (1, 2, 3)]
    for f in range(12):
        b.step(seqs, [s.frame(f) for s in syn])
        b.check(seqs, f"frame {f}")


def test_fresh_and_reset_handles_join_mid_run(product, cfg_dir, bed):
    """A fresh handle runs its first frame beside handles in steady state; a handle reset between steps takes the next
    recording in its slot (its first frame again) while the others go on."""
    b, seqs = bed["bed"], bed["seqs"]
    syn = {1: Synth(1, 21), 2: Synth(2, 22), 3: Synth(3, 23), 5: Synth(1, 25)}
    seqs += [synth_seq(product, cfg_dir, 1), synth_seq(product, cfg_dir, 2), synth_seq(product, cfg_dir, 3)]
    start = {0: (1, 0), 1: (2, 0)}  # slot -> (recording, step it started at)
    for f in range(10):
        if f == 3:
            start[2] = (3, f)  # the fresh C3 handle joins
        if f == 6:
            seqs[0].reset()  # slot 0 takes the next C1 recording
            start[0] = (5, f)
        active = sorted(start)
        b.step([seqs[s] for s in active], [syn[start[s][0]].frame(f - start[s][1]) for s in active])
        b.check([seqs[s] for s in active], f"step {f}")
        if f == 3:
            assert seqs[2].gpu.counts()["TWO_FRAMES"] == 0 and seqs[0].gpu.counts()["TWO_FRAMES"] == 1


def test_method_1_beside_method_2(product, cfg_dir, tmp_path, bed):
    b, seqs = bed["bed"], bed["seqs"]
    syn = [Synth(1, 31), Synth(1, 32), Synth(2, 33), Synth(2, 34)]
    m1 = {sc: write_cfg(tmp_path, f"m1_{sc}.txt", base=cfg_dir / CONFIGS[sc], method_choice=1) for sc in (1, 2)}
    seqs += [synth_seq(product, cfg_dir, 1, m1[1]), synth_seq(product, cfg_dir, 1), synth_seq(product, cfg_dir, 2),
             synth_seq(product, cfg_dir, 2, m1[2], n_bad=2, n_good=5)]
    for f in range(8):
        b.step(seqs, [s.frame(f) for s in syn])
        b.check(seqs, f"frame {f}")


def test_crop_beside_voxel_ground_modes(product, cfg_dir, tmp_path, bed):
    """C4 terrain in the crop mode, ground_mode 1 and ground_mode 2, beside a C1 frame: the ground stage runs over the two
    voxel-mode sequences only (9 launches), then one frame launch, then one gather for the one handle with records."""
    b, seqs = bed["bed"], bed["seqs"]
    terrain = cfg_dir / CONFIGS[4]
    cfgs = [write_cfg(tmp_path, "crop.txt", base=terrain, ground_mode=0), write_cfg(tmp_path, "g1.txt", base=terrain, ground_mode=1),
            terrain, cfg_dir / CONFIGS[1]]
    syn = [Synth(4, 41), Synth(4, 42), Synth(4, 43), Synth(1, 44)]
    seqs += [Seq(product, c, s.max_points, max_cells=C4_CELLS) for c, s in zip(cfgs[:3], syn)]
    seqs.append(Seq(product, cfgs[3], syn[3].max_points, step=22, out_records=True))
    for f in range(6):
        before = [q.gpu.launch_count() for q in seqs]
        b.step(seqs, [s.frame(f) for s in syn])
        after = [q.gpu.launch_count() for q in seqs]
        assert after[0] - before[0] == 9 + 1 + 1 and after[1:] == before[1:], (before, after)
        b.check(seqs, f"frame {f}")
        assert all(q.gpu.counts()["NG"] > 0 for q in seqs[1:3])


def test_large_k_beside_default_handles(product, cfg_dir, tmp_path, bed):
    """A handle with max_clusters above 16,384 on the lattice scene at K = 16,385 (the large-K path) beside default handles:
    the launch runs the LK kernel for every sequence, which leaves the small frames exact."""
    b, seqs = bed["bed"], bed["seqs"]
    frames = scene_frames(16_385)
    lattice = Seq(product, scene_cfg(tmp_path), max(len(p) for p in frames), n_bad=N_BAD, n_good=N_GOOD, max_clusters=MAX_CLUSTERS)
    syn = [Synth(1, 51), Synth(2, 52)]
    seqs += [synth_seq(product, cfg_dir, 1), lattice, synth_seq(product, cfg_dir, 2)]
    for f in range(len(frames)):
        b.step(seqs, [syn[0].frame(f), (frames[f], IDENTITY_POSE), syn[1].frame(f)])
        b.check(seqs, f"frame {f}")
        assert lattice.gpu.counts()["K"] == 16_385
    assert lattice.gpu.tap("cluster_removed").sum() > 0


def test_output_records_for_some_handles(product, cfg_dir, bed):
    """Output records on for three handles (16-, 22- and 32-byte records) and off for two (22 and 32 bytes in, PointXYZI
    out)."""
    b, seqs = bed["bed"], bed["seqs"]
    plan = [(1, 16, True), (2, 22, True), (3, 32, True), (1, 22, False), (2, 32, False)]
    syn = [Synth(sc, 60 + i) for i, (sc, _, _) in enumerate(plan)]
    seqs += [synth_seq(product, cfg_dir, sc, step=step, out_records=rec) for sc, step, rec in plan]
    for f in range(6):
        before = seqs[0].gpu.launch_count()
        b.step(seqs, [s.frame(f) for s in syn])
        assert seqs[0].gpu.launch_count() - before == 2
        b.check(seqs, f"frame {f}")


@pytest.mark.parametrize("S", [1, 37, 160])
def test_batch_widths(product, cfg_dir, tmp_path, bed, S):
    """S = 1, 37 and 160 (more sequences than CTAs: longest frames first onto the least-loaded CTA). C1 sequences with
    method 1 or 2 and with or without 22-byte output records, a few C2 ones, and frames cut to different lengths."""
    b, seqs = bed["bed"], bed["seqs"]
    m1 = write_cfg(tmp_path, "m1.txt", base=cfg_dir / CONFIGS[1], method_choice=1)
    kinds = []
    for s in range(S):
        if s % 9 == 4:
            kinds.append((2, None, 16, False))
        else:
            kinds.append((1, m1 if s % 3 == 1 else None, 22 if s % 3 == 2 else 16, s % 3 == 2))
    syn = {sc: [Synth(sc, 70 + k) for k in range(4)] for sc in (1, 2)}
    seqs += [synth_seq(product, cfg_dir, sc, cfg, step=step, out_records=rec) for sc, cfg, step, rec in kinds]
    for f in range(4):
        data = {(sc, k): syn[sc][k].frame(f) for sc in (1, 2) for k in range(4)}
        frames = []
        for s, (sc, _, _, _) in enumerate(kinds):
            pts, pose = data[(sc, s % 4)]
            frames.append((np.ascontiguousarray(pts[: len(pts) * (1 + s % 4) // 4]), pose))
        b.step(seqs, frames)
        b.check(seqs, f"frame {f}")


def test_capacity_errors_stay_in_their_sequence(product, cfg_dir, bed):
    """A frame whose ground grid exceeds max_cells raises ERR_GROUND_CAP in its own sequence's counts only; a frame above
    its handle's max_points refuses the step with MOR_ERR_CAPACITY naming that sequence, changes no handle, and the
    steps after it stay exact in every sequence."""
    b, seqs = bed["bed"], bed["seqs"]
    syn = [Synth(4, 81), Synth(1, 82), Synth(2, 83)]
    seqs += [Seq(product, cfg_dir / CONFIGS[4], syn[0].max_points + 1, max_cells=1 << 20), synth_seq(product, cfg_dir, 1),
             synth_seq(product, cfg_dir, 2)]
    for f in range(6):
        frames = [s.frame(f) for s in syn]
        if f == 2:  # one point at z = 1e3: the ground grid's box needs more than max_cells cells
            pts, pose = frames[0]
            frames[0] = (np.ascontiguousarray(np.concatenate([pts, np.float32([[1.0, 1.0, 1e3, 0.5]])])), pose)
        if f == 4:  # one point more than the C1 handle's max_points
            pts, pose = frames[1]
            big = np.ascontiguousarray(np.concatenate([pts, np.zeros((seqs[1].maxp + 1 - len(pts), 4), np.float32)]))
            counts = [q.gpu.counts() for q in seqs]
            with pytest.raises(MorError) as e:
                b.step(seqs, [frames[0], (big, pose), frames[2]], twins=False)
            assert e.value.status == ERR_CAPACITY and "sequence 1" in str(e.value) and "max_points" in str(e.value), str(e.value)
            assert [q.gpu.counts() for q in seqs] == counts
        b.step(seqs, frames)
        b.check(seqs, f"frame {f}")
        errs = [q.gpu.counts()["ERRFLAGS"] for q in seqs]
        assert errs[1:] == [0, 0] and (errs[0] & ERR_GROUND_CAP if f == 2 else f > 2 or errs[0] == 0), (f, errs)


def test_refused_steps_leave_every_handle_steppable(product, cfg_dir, bed):
    """A duplicate handle, a handle with submitted frames in flight and a handle with kernel profiling on are each
    MOR_ERR_ARG naming the rule; the step after each refusal (rule lifted) is exact in every sequence."""
    b, seqs = bed["bed"], bed["seqs"]
    syn = [Synth(1, 91), Synth(2, 92), Synth(3, 93)]
    seqs += [synth_seq(product, cfg_dir, sc) for sc in (1, 2, 3)]
    f = 0

    def good_step():
        nonlocal f
        b.step(seqs, [s.frame(f) for s in syn])
        b.check(seqs, f"frame {f}")
        f += 1

    def refused(hs, frames, rule):
        launches = [q.gpu.launch_count() for q in seqs]
        with pytest.raises(MorError) as e:
            b.step(hs, frames, twins=False)
        assert e.value.status == ERR_ARG and rule in str(e.value), str(e.value)
        assert [q.gpu.launch_count() for q in seqs] == launches

    good_step()
    good_step()
    refused([seqs[0], seqs[1], seqs[0]], [s.frame(f) for s in (syn[0], syn[1], syn[0])], "appears twice")
    good_step()
    # a frame of sequence 1 submitted and not collected: in flight
    pts, pose = syn[1].frame(f)
    out = np.empty((len(pts), 8), np.float32)
    seqs[1].gpu.submit_frame(pts, pose, out)
    refused(seqs, [s.frame(f + 1) for s in syn], "in flight")
    got = seqs[1].gpu.collect_frame().copy()
    seqs[1].twin.push_raw_cloud_and_pose(pts, pose)
    assert got.tobytes() == seqs[1].twin.filter_cloud().tobytes()
    f += 1
    for s in (0, 2):  # the other two take the same frame alone, so that all three go on in step
        p, q = syn[s].frame(f - 1)
        for h in (seqs[s].gpu, seqs[s].twin):
            h.push_raw_cloud_and_pose(p, q)
            h.filter_cloud()
    good_step()
    seqs[2].gpu.set_kernel_profiling(True)
    refused(seqs, [s.frame(f) for s in syn], "profiling")
    seqs[2].gpu.set_kernel_profiling(False)
    good_step()
    good_step()
