"""mor_set_pipelining for the voxel ground modes and method 1 (-m gpu): the pipelined launch variants k_frame_pipe_ground,
k_frame_pipe_pde and k_frame_pipe_ground_pde must deliver what one kernel per frame delivers, byte for byte, and what the
oracle delivers, on the streaming and device-resident paths, with and without output records, and when pipelined launches
are mixed with every other call of the protocol."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from dynamicslamtool_b200 import MorError, MovingObjectRemoval, SequenceBatch, Synth
from helpers import ROOT, crc, write_cfg
from parity import ParityStats, compare_frame
from records_ref import expected_records, make_records

pytestmark = pytest.mark.gpu

CASES = {  # name -> (scenario, base config, overrides, frames)
    "c4_ground1": (4, "MOR_config_terrain.txt", {"ground_mode": 1}, 8),
    "c4_ground2": (4, "MOR_config_terrain.txt", {"ground_mode": 2}, 8),
    "c1_method1": (1, "MOR_config.txt", {"method_choice": 1}, 16),
    "hdl64_method1": (2, "MOR_config_hdl64.txt", {"method_choice": 1}, 12),
    "c4_ground2_method1": (4, "MOR_config_terrain.txt", {"ground_mode": 2, "method_choice": 1}, 8),
}
GROUND_CASES = ("c4_ground1", "c4_ground2", "c4_ground2_method1")
ERR_CAPACITY = 6
DEPTH = 4  # MOR_STREAM_DEPTH


def _setup(cfg_dir, tmp_path, case, frames=None):
    scenario, base, ov, n = CASES[case]
    cfg = write_cfg(tmp_path, base=cfg_dir / base, **ov)
    s = Synth(scenario, scenario)
    return cfg, s, [s.frame(f) for f in range(frames or n)]


def _handle(product, cfg, maxp, pipelining, max_cells=1 << 21):
    h = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=maxp, max_cells=max_cells)
    h.set_pipelining(pipelining)
    return h


def _alloc(product, nbytes):
    p = C.c_void_p()
    assert product.device_alloc(0, max(nbytes, 16), C.byref(p)) == 0
    return p


def _upload(product, d, a):
    if a.nbytes:
        assert product.device_upload(0, d, a.ctypes.data_as(C.c_void_p), a.nbytes) == 0


def _download(product, d, n, step=None):
    out = np.empty((n, step), np.uint8) if step else np.empty((n, 8), np.float32)
    if n:
        assert product.device_download(0, out.ctypes.data_as(C.c_void_p), C.c_void_p(d), out.nbytes) == 0
    return out


def _pinned(product, shape, dtype, keep):
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    assert product.alloc_pinned(nbytes, C.byref(p)) == 0
    keep.append(p)
    return np.frombuffer((C.c_uint8 * nbytes).from_address(p.value), dtype=dtype).reshape(shape)


def _device_output(product, h):
    return _download(product, h.output_device(), h.counts()["NOUT"])


@pytest.mark.parametrize("case", list(CASES))
def test_streamed_frames_equal_unpipelined_and_oracle(product, oracle, cfg_dir, tmp_path, case):
    cfg, s, seq = _setup(cfg_dir, tmp_path, case)
    maxp = s.max_points
    ref = _handle(product, cfg, maxp, False)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    want, want_orc = [], []
    for pts, pose in seq:
        ref.push_raw_cloud_and_pose(pts, pose)
        want.append(crc(ref.filter_cloud()))
        orc.push_raw_cloud_and_pose(pts, pose)
        want_orc.append(crc(orc.filter_cloud()))
    assert want == want_orc
    m = _handle(product, cfg, maxp, True)
    keep = []
    ins = [_pinned(product, (maxp, 4), np.float32, keep) for _ in range(DEPTH)]
    outs = [_pinned(product, (maxp, 8), np.float32, keep) for _ in range(DEPTH)]
    got = []
    for f, (pts, pose) in enumerate(seq):
        ins[f % DEPTH][: len(pts)] = pts
        m.submit_frame(ins[f % DEPTH][: len(pts)], pose, outs[f % DEPTH])
        if f >= DEPTH - 1:
            got.append(crc(m.collect_frame()))
    while m.frames_in_flight():
        got.append(crc(m.collect_frame()))
    assert got == want
    for tap in ("mo_conf", "mo_centroids"):
        assert np.array_equal(m.tap(tap), ref.tap(tap)) and np.array_equal(m.tap(tap), orc.tap(tap)), tap
    m.close()
    for p in keep:
        product.free_pinned(p)


@pytest.mark.parametrize("case", list(CASES))
def test_device_resident_pipelined_frames_match_oracle(product, oracle, cfg_dir, tmp_path, case):
    """push_device + filter_device(None, 0, want_count=False): the back half of frame f waits for the front half of f+1.
    At the checkpoints (the comparison makes the pending back half run alone) every tap is held to the oracle."""
    cfg, s, seq = _setup(cfg_dir, tmp_path, case)
    maxp = s.max_points
    pipe = _handle(product, cfg, maxp, True)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    d = [_alloc(product, maxp * 16) for _ in seq]
    for f, (pts, _) in enumerate(seq):
        _upload(product, d[f], pts)
    stats = ParityStats()
    frames = len(seq)
    checkpoints = {0, 1, 2, 5, frames - 2, frames - 1}
    for f, (pts, pose) in enumerate(seq):
        pipe.push_device(d[f].value, len(pts), pose)
        pipe.filter_device(None, 0, want_count=False)
        orc.push_raw_cloud_and_pose(pts, pose)
        oo = orc.filter_cloud().copy()
        if f in checkpoints:
            bad = compare_frame(pipe, orc, _device_output(product, pipe), oo, stats)
            assert not bad, f"frame {f}: {bad}"
    assert stats.matches > 0
    pipe.close()
    for p in d:
        product.device_free(0, p)


@pytest.mark.parametrize("case", list(CASES))
def test_pipelined_output_records_equal_oracle(product, oracle, cfg_dir, tmp_path, case):
    """22-byte XYZIRT records: device-resident (one input buffer per frame: a frame's records are gathered when its back
    half runs) and streaming; every frame's records equal those the oracle's bookkeeping selects."""
    cfg, s, seq = _setup(cfg_dir, tmp_path, case, frames=6)
    maxp = s.max_points
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    recs, want = [], []
    for pts, pose in seq:
        rec, step, offs = make_records(pts, "xyzirt22")
        orc.push_raw_cloud_and_pose(rec, pose, point_step=step, offsets=offs)
        orc.filter_cloud()
        recs.append(rec)
        want.append(expected_records(orc, rec).tobytes())
    # device-resident
    dev = _handle(product, cfg, maxp, True)
    dev.set_output_records(True)
    d_in = [_alloc(product, maxp * 32) for _ in seq]
    for f, (rec, (_, pose)) in enumerate(zip(recs, seq)):
        _upload(product, d_in[f], rec)
        dev.push_device(d_in[f].value, len(rec), pose, step, offs)
        dev.filter_device(None, 0, want_count=False)
        if f % 2 == 1:  # (every other frame is read back, which runs its back half alone)
            got = _download(product, dev.output_device(), dev.counts()["NOUT"], step)
            assert got.tobytes() == want[f], f"device path frame {f}"
    got = _download(product, dev.output_device(), dev.counts()["NOUT"], step)
    assert got.tobytes() == want[-1]
    # streaming
    st = _handle(product, cfg, maxp, True)
    st.set_output_records(True)
    keep = []
    ins = [_pinned(product, (maxp, step), np.uint8, keep) for _ in range(DEPTH)]
    outs = [_pinned(product, (maxp, step), np.uint8, keep) for _ in range(DEPTH)]
    got = []
    for f, (rec, (_, pose)) in enumerate(zip(recs, seq)):
        ins[f % DEPTH][: len(rec)] = rec
        st.submit_frame(ins[f % DEPTH][: len(rec)], pose, outs[f % DEPTH], point_step=step, offsets=offs)
        if f >= DEPTH - 1:
            got.append(st.collect_frame().tobytes())
    while st.frames_in_flight():
        got.append(st.collect_frame().tobytes())
    assert got == want
    for h in (dev, st):
        h.close()
    for p in d_in:
        product.device_free(0, p)
    for p in keep:
        product.free_pinned(p)


@pytest.mark.parametrize("records", [False, True])
@pytest.mark.parametrize("case", ["c4_ground1", "c1_method1", "c4_ground2_method1"])
def test_pipelined_launch_counts(product, cfg_dir, tmp_path, case, records):
    """Per device-resident push: 9 ground launches + 1 pipelined launch (voxel ground modes), 1 (method 1 with the crop
    mode); record mode adds the gather of the back half that ran; a flush adds the back half alone (+ its gather)."""
    cfg, s, seq = _setup(cfg_dir, tmp_path, case, frames=4)
    h = _handle(product, cfg, s.max_points, True)
    h.set_output_records(records)
    d = [_alloc(product, s.max_points * 16) for _ in seq]
    base = 10 if case in GROUND_CASES else 1
    for f, (pts, pose) in enumerate(seq):
        _upload(product, d[f], pts)
        before = h.launch_count()
        h.push_device(d[f].value, len(pts), pose)
        h.filter_device(None, 0, want_count=False)
        assert h.launch_count() - before == base + (1 if records and f > 0 else 0), f"push {f}"
    before = h.launch_count()
    h.counts()  # the pending back half runs alone
    assert h.launch_count() - before == 1 + (1 if records else 0)
    h.close()
    for p in d:
        product.device_free(0, p)


def _protocol_run(product, cfg, seq, maxp, pipelining):
    """A device-resident run that mixes pipelined launches with every other call; returns what it observed."""
    h = _handle(product, cfg, maxp, pipelining)
    d = [_alloc(product, maxp * 16) for _ in seq]
    for f, (pts, _) in enumerate(seq):
        _upload(product, d[f], pts)
    d_out = _alloc(product, maxp * 32)
    seen = []

    def snap(tag):
        seen.append((tag, h.counts(), _device_output(product, h).tobytes(), h.tap("mo_conf").tobytes(), h.tap("mo_centroids").tobytes(),
                     h.tap("removed_mask").tobytes()))

    def step(f, filt=True):
        h.push_device(d[f].value, len(seq[f][0]), seq[f][1])
        if filt:
            h.filter_device(None, 0, want_count=False)

    step(0); step(1)
    step(2, filt=False)                              # a push that is never filtered
    step(3)
    n = h.filter_device(d_out.value, maxp)            # a second filter call on the same frame
    h.sync()
    seen.append(("double filter", n, _download(product, d_out.value, n).tobytes()))
    step(4)
    h.set_pipelining(False)                           # toggled off ...
    step(5); snap("after toggle off")
    h.set_pipelining(pipelining)                      # ... and back on
    step(6); step(7)
    h.reset()                                         # reset in the middle of the run
    step(8); step(9); snap("after reset")
    step(10)
    h.set_kernel_profiling(True)                      # one kernel per phase
    step(11); snap("profiled")
    h.set_kernel_profiling(False)
    step(12)
    SequenceBatch([h]).step_device([d[13].value], [len(seq[13][0])], [seq[13][1]], [d_out.value])  # takes in the pending back half
    h.sync()
    seen.append(("batched", h.counts(), _download(product, d_out.value, h.counts()["NOUT"]).tobytes()))
    step(14)
    h.push_device(d[15].value, 0, seq[15][1]); h.filter_device(None, 0, want_count=False)  # an empty frame
    h.push_device(d[16].value, 300, seq[16][1]); h.filter_device(None, 0, want_count=False)  # 300 points
    step(17); step(18)
    snap("end")
    h.close()
    for p in d + [d_out]:
        product.device_free(0, p)
    return seen


@pytest.mark.parametrize("case", list(CASES))
def test_protocol_mixing_equals_unpipelined(product, cfg_dir, tmp_path, case):
    cfg, s, seq = _setup(cfg_dir, tmp_path, case, frames=19)
    a = _protocol_run(product, cfg, seq, s.max_points, True)
    b = _protocol_run(product, cfg, seq, s.max_points, False)
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x == y, f"{x[0]}: differs from the unpipelined handle"


@pytest.mark.parametrize("case", GROUND_CASES)
def test_ground_capacity_error_is_reported_for_its_frame(product, cfg_dir, tmp_path, case):
    """One point at z = 1e3 needs more than max_cells cells: ERR_GROUND_CAP for that frame on the streaming and the
    device paths with pipelining; the frames after it equal those of an unpipelined handle."""
    bad = 2
    cfg, s, seq = _setup(cfg_dir, tmp_path, case, frames=6)
    maxp = s.max_points + 1
    seq = [(np.ascontiguousarray(np.concatenate([p, np.float32([[1.0, 1.0, 1e3, 0.5]])])) if f == bad else p, pose)
           for f, (p, pose) in enumerate(seq)]
    # streaming
    hs = {m: _handle(product, cfg, maxp, m, max_cells=1 << 20) for m in (False, True)}
    keep = []
    got = {}
    for m, h in hs.items():
        ins = [_pinned(product, (maxp, 4), np.float32, keep) for _ in range(DEPTH)]
        outs = [_pinned(product, (maxp, 8), np.float32, keep) for _ in range(DEPTH)]
        res = []

        def collect():
            try:
                res.append(crc(h.collect_frame()))
            except MorError as e:
                assert e.status == ERR_CAPACITY, e
                res.append("capacity")

        for f, (pts, pose) in enumerate(seq):
            if h.frames_in_flight() == DEPTH:
                collect()
            ins[f % DEPTH][: len(pts)] = pts
            h.submit_frame(ins[f % DEPTH][: len(pts)], pose, outs[f % DEPTH])
        while h.frames_in_flight():
            collect()
        got[m] = res
        h.close()
    assert got[True] == got[False] and [f for f, v in enumerate(got[True]) if v == "capacity"] == [bad]
    # device-resident
    hs = {m: _handle(product, cfg, maxp, m, max_cells=1 << 20) for m in (False, True)}
    d = [_alloc(product, maxp * 16) for _ in seq]
    for f, (pts, _) in enumerate(seq):
        _upload(product, d[f], pts)
    for f, (pts, pose) in enumerate(seq):
        for m, h in hs.items():
            h.push_device(d[f].value, len(pts), pose)
            if f == bad:
                with pytest.raises(MorError) as e:
                    h.filter_device(None, 0)
                assert e.value.status == ERR_CAPACITY and h.counts()["ERRFLAGS"] & 8
            else:
                h.filter_device(None, 0, want_count=False)
    a, b = hs[True], hs[False]
    assert a.counts() == b.counts() and _device_output(product, a).tobytes() == _device_output(product, b).tobytes()
    assert a.tap("mo_conf").tobytes() == b.tap("mo_conf").tobytes()
    for h in hs.values():
        h.close()
    for p in d:
        product.device_free(0, p)
    for p in keep:
        product.free_pinned(p)


@pytest.mark.parametrize("case", ["c4_ground2", "c1_method1"])
def test_harness_stream_replay_writes_the_same_files(built, cfg_dir, tmp_path, case):
    """mov_harness --replay ... --out with --stream (pipelined launches) writes files byte-identical to the callback loop."""
    from test_gpu_harness import _write_replay_dir
    exe = ROOT / "harness" / "mov_harness"
    if not exe.exists():
        subprocess.check_call(["make", "-C", str(ROOT / "harness")])
    cfg, _, seq = _setup(cfg_dir, tmp_path, case, frames=9)
    rec = tmp_path / "rec"
    _write_replay_dir(rec, seq, 7)
    outs = []
    for extra in ([], ["--stream"]):
        out = tmp_path / ("out_stream" if extra else "out")
        out.mkdir()
        res = subprocess.run([str(exe), str(cfg), "--replay", str(rec), "--out", str(out)] + extra, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr
        outs.append({p.name: p.read_bytes() for p in sorted(out.iterdir())})
    assert len(outs[0]) == len(seq) and outs[0] == outs[1]
