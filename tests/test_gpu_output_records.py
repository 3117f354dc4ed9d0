"""Output records (mor_set_output_records, -m gpu): on every output path the GPU delivers, byte for byte, the input records
the oracle's bookkeeping selects (tests/records_ref.py), and the PointXYZI output of the default mode is untouched."""
import ctypes as C

import numpy as np
import pytest

from dynamicslamtool_b200 import MorError, MovingObjectRemoval, SequenceBatch, Synth
from helpers import write_cfg
from parity import compare_frame
from records_ref import LAYOUTS, expected_records, make_records

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_CAPACITY, ERR_STATE = 5, 6, 8


def _alloc(product, nbytes):
    p = C.c_void_p()
    assert product.device_alloc(0, max(nbytes, 16), C.byref(p)) == 0
    return p


def _upload(product, d, a):
    if a.nbytes:
        assert product.device_upload(0, d, a.ctypes.data_as(C.c_void_p), a.nbytes) == 0


def _download(product, d, n, step):
    out = np.empty((n, step), np.uint8)
    if n:
        assert product.device_download(0, out.ctypes.data_as(C.c_void_p), C.c_void_p(d), n * step) == 0
    return out


def _pinned(product, shape, dtype):
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    assert product.alloc_pinned(nbytes, C.byref(p)) == 0
    buf = (C.c_uint8 * nbytes).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape), p


def _frames(scenario, seed, idx):
    s = Synth(scenario, seed)
    return s, [s.frame(f) for f in idx]


CASES = [  # (scenario, config, overrides, frame indices)
    (1, "MOR_config.txt", {}, range(8)),
    (2, "MOR_config_hdl64.txt", {}, range(98, 108)),  # C2 including its dense frames 101-107
    (4, "MOR_config_terrain.txt", {"ground_mode": 1}, range(5)),
    (4, "MOR_config_terrain.txt", {"ground_mode": 2}, range(5)),
    (1, "MOR_config.txt", {"method_choice": 1}, range(8)),
]


@pytest.mark.parametrize("case", range(len(CASES)))
@pytest.mark.parametrize("layout", ["xyzirt22", "xyzi16", "odd13", "odd19", "xyz12"])
def test_host_path_records_equal_oracle(product, oracle, cfg_dir, tmp_path, case, layout):
    """mor_filter_cloud in record mode, a repeated filter call on some frames (k_filter_again), and a PointXYZI twin that
    never had the mode on: its output and taps equal those of the oracle as before."""
    scenario, base, ov, idx = CASES[case]
    if layout != "xyzirt22" and case not in (0, 1):
        pytest.skip("every layout on C1 / C2; the other cases with the velodyne record")
    cfg = write_cfg(tmp_path, base=cfg_dir / base, **ov)
    s, seq = _frames(scenario, scenario, idx)
    kw = dict(binding=product, max_points=s.max_points, max_cells=1 << 21)
    gpu, twin = MovingObjectRemoval(cfg, 4, 3, **kw), MovingObjectRemoval(cfg, 4, 3, **kw)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    gpu.set_output_records(True)
    for f, (pts, pose) in enumerate(seq):
        rec, step, offs = make_records(pts, layout)
        for m in (gpu, twin, orc):
            m.push_raw_cloud_and_pose(rec, pose, point_step=step, offsets=offs)
        for rep in range(2 if f % 3 == 2 else 1):
            og, ot, oo = gpu.filter_cloud().copy(), twin.filter_cloud().copy(), orc.filter_cloud().copy()
            assert og.dtype == np.uint8 and og.shape == (len(oo), step)
            assert og.tobytes() == expected_records(orc, rec).tobytes(), f"frame {f} call {rep}: records differ"
            if rep == 0:
                assert not compare_frame(twin, orc, ot, oo)
            else:  # (a repeated call only ever adds to the removal mask: compare the output alone)
                assert ot.tobytes() == oo.tobytes()
            for tap in ("removed_mask", "point_class", "mo_conf"):
                assert gpu.tap(tap).tobytes() == twin.tap(tap).tobytes(), f"frame {f}: {tap}"


@pytest.mark.parametrize("path", ["device", "zero_copy", "pipelined"])
@pytest.mark.parametrize("layout", ["xyzirt22", "xyzi16", "odd13"])
def test_device_paths_records_equal_oracle(product, oracle, cfg_dir, path, layout):
    s, seq = _frames(1, 3, range(10))
    cfg = cfg_dir / "MOR_config.txt"
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=s.max_points)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    gpu.set_output_records(True)
    gpu.set_pipelining(path == "pipelined")
    step = LAYOUTS[layout][0]
    # pipelined: a frame's records are gathered when its back half runs (with the next push): one input buffer per frame
    d_in = [_alloc(product, s.max_points * 32) for _ in seq]
    d_out = _alloc(product, s.max_points * 32)
    try:
        for f, (pts, pose) in enumerate(seq):
            rec, step, offs = make_records(pts, layout)
            _upload(product, d_in[f], rec)
            gpu.push_device(d_in[f].value, len(rec), pose, step, offs)
            orc.push_raw_cloud_and_pose(rec, pose, point_step=step, offsets=offs)
            orc.filter_cloud()
            want = expected_records(orc, rec)
            if path == "device":
                n = gpu.filter_device(d_out.value, s.max_points)
                gpu.sync()  # (the device-to-device copy runs on the handle's stream)
                got = _download(product, d_out.value, n, step)
            elif path == "zero_copy":
                n = gpu.filter_device(None, 0)
                got = _download(product, gpu.output_device(), n, step)
            else:
                gpu.filter_device(None, 0, want_count=False)  # the back half stays pending until the next push
                if f != len(seq) - 1:
                    continue
                gpu.sync()
                n = gpu.counts()["NOUT"]
                got = _download(product, gpu.output_device(), n, step)
            assert got.tobytes() == want.tobytes(), f"{path} frame {f}"
        assert np.array_equal(gpu.tap("mo_conf"), orc.tap("mo_conf"))
    finally:
        for p in d_in + [d_out]:
            product.device_free(0, p)


@pytest.mark.parametrize("scenario,cfg,frames,pipelining,layout", [
    (1, "MOR_config.txt", 16, False, "xyzirt22"), (1, "MOR_config.txt", 16, True, "xyzirt22"),
    (2, "MOR_config_hdl64.txt", 12, True, "xyzi16"), (2, "MOR_config_hdl64.txt", 12, False, "odd19")])
def test_streaming_records_equal_oracle(product, oracle, cfg_dir, scenario, cfg, frames, pipelining, layout):
    s, seq = _frames(scenario, scenario, range(frames))
    m = MovingObjectRemoval(cfg_dir / cfg, 4, 3, binding=product, max_points=s.max_points)
    orc = MovingObjectRemoval(cfg_dir / cfg, 4, 3, binding=oracle)
    m.set_output_records(True)
    m.set_pipelining(pipelining)
    step = LAYOUTS[layout][0]
    want = []
    for pts, pose in seq:
        rec, step, offs = make_records(pts, layout)
        orc.push_raw_cloud_and_pose(rec, pose, point_step=step, offsets=offs)
        orc.filter_cloud()
        want.append(expected_records(orc, rec).tobytes())
    DEPTH, keep, ins, outs = 4, [], [], []
    for _ in range(DEPTH):
        a, pa = _pinned(product, (s.max_points, step), np.uint8)
        o, po = _pinned(product, (s.max_points, step), np.uint8)
        ins.append(a); outs.append(o); keep += [pa, po]
    got = []
    try:
        for f, (pts, pose) in enumerate(seq):
            rec, step, offs = make_records(pts, layout)
            ins[f % DEPTH][: len(rec)] = rec
            m.submit_frame(ins[f % DEPTH][: len(rec)], pose, outs[f % DEPTH], point_step=step, offsets=offs)
            if f == 0:
                with pytest.raises(MorError) as e:
                    m.set_output_records(False)
                assert e.value.status == ERR_STATE
            if f >= DEPTH - 1:
                got.append(m.collect_frame().tobytes())
        while m.frames_in_flight():
            got.append(m.collect_frame().tobytes())
        assert got == want
    finally:
        for p in keep:
            product.free_pinned(p)


@pytest.mark.parametrize("S,base,ov", [(3, "MOR_config.txt", {}), (37, "MOR_config.txt", {}),
                                        (3, "MOR_config_terrain.txt", {"ground_mode": 1})])
def test_batched_records_equal_oracle_and_unbatched(product, oracle, cfg_dir, tmp_path, S, base, ov):
    """Batched steps with a mix of empty, small and full frames; the 22-byte record. Each sequence matches its oracle
    (S = 3) or an unbatched record-mode twin (every sequence) byte for byte; d_out[s] is exactly n[s] records long."""
    cfg = write_cfg(tmp_path, base=cfg_dir / base, **ov)
    scen = 4 if ov else 1
    syn = [Synth(scen, 60 + s % 8) for s in range(S)]
    maxp = syn[0].max_points
    kw = dict(binding=product, max_points=maxp, max_cells=1 << 21)
    gpus, twins = [MovingObjectRemoval(cfg, 4, 3, **kw) for _ in range(S)], [MovingObjectRemoval(cfg, 4, 3, **kw) for _ in range(S)]
    orcs = [MovingObjectRemoval(cfg, 4, 3, binding=oracle) for _ in range(S)] if S <= 3 else []
    for g in gpus + twins:
        g.set_output_records(True)
    batch = SequenceBatch(gpus)
    step, offs = 22, LAYOUTS["xyzirt22"][1]
    d_in = [_alloc(product, maxp * 32) for _ in range(S)]
    d_out = [_alloc(product, maxp * step + 64) for _ in range(S)]
    d_tout = [_alloc(product, maxp * step) for _ in range(S)]
    guard = np.full(64, 0x3C, np.uint8)
    try:
        for f in range(5):
            recs, ns, poses = [], [], []
            for s in range(S):
                pts, pose = syn[s].frame(f)
                kind = (s + f) % 3  # 0 empty, 1 small, 2 full
                pts = pts[:0] if kind == 0 else pts[:300] if kind == 1 else pts
                rec, _, _ = make_records(np.ascontiguousarray(pts), "xyzirt22")
                recs.append(rec); ns.append(len(rec)); poses.append(pose)
                _upload(product, d_in[s], rec)
                # guard bytes right behind the n[s] records: the batched gather must not write past them
                assert product.device_upload(0, C.c_void_p(d_out[s].value + len(rec) * step), guard.ctypes.data_as(C.c_void_p), 64) == 0
            for g in gpus + twins:
                g.sync()
            batch.step_device([p.value for p in d_in], ns, poses, [p.value for p in d_out], step, offs)
            for s in range(S):
                twins[s].push_device(d_in[s].value, ns[s], poses[s], step, offs)
                twins[s].filter_device(d_tout[s].value, maxp)
                twins[s].sync()
            for s in range(S):
                gpus[s].sync()
                n = gpus[s].counts()["NOUT"]
                got = _download(product, d_out[s].value, n, step)
                tail = np.empty(64, np.uint8)
                assert product.device_download(0, tail.ctypes.data_as(C.c_void_p), C.c_void_p(d_out[s].value + ns[s] * step), 64) == 0
                assert np.array_equal(tail, guard), f"sequence {s} frame {f}: bytes written past n[s] records"
                assert got.tobytes() == _download(product, d_tout[s].value, twins[s].counts()["NOUT"], step).tobytes()
                assert gpus[s].output_device() == d_out[s].value
                if orcs:
                    orcs[s].push_raw_cloud_and_pose(recs[s], poses[s], point_step=step, offsets=offs)
                    orcs[s].filter_cloud()
                    assert got.tobytes() == expected_records(orcs[s], recs[s]).tobytes(), f"sequence {s} frame {f}"
    finally:
        for p in d_in + d_out + d_tout:
            product.device_free(0, p)


def test_errors_launch_count_toggle_and_reset(product, oracle, cfg_dir):
    cfg = cfg_dir / "MOR_config.txt"
    s, seq = _frames(1, 7, range(6))
    maxp = s.max_points
    on, off, never = (MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=maxp) for _ in range(3))
    on.set_output_records(True)
    off.set_output_records(True)
    off.set_output_records(False)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    for pts, pose in seq:
        rec, step, offs = make_records(pts, "xyzirt22")
        counts0 = [m.launch_count() for m in (on, off, never)]
        for m in (on, off, never, orc):
            m.push_raw_cloud_and_pose(rec, pose, point_step=step, offsets=offs)
        oo = orc.filter_cloud().copy()
        assert on.filter_cloud().tobytes() == expected_records(orc, rec).tobytes()
        assert off.filter_cloud().tobytes() == never.filter_cloud().tobytes() == oo.tobytes()
        d = [m.launch_count() - c for m, c in zip((on, off, never), counts0)]
        assert d[0] == d[2] + 1 and d[1] == d[2]  # one gather per frame in record mode, nothing otherwise
    # toggling between frames: XYZI frames stay identical to the never-toggled handle
    on.set_output_records(False)
    pts, pose = s.frame(6)
    on.push_raw_cloud_and_pose(pts, pose)
    never.push_raw_cloud_and_pose(pts, pose)
    assert on.filter_cloud().tobytes() == never.filter_cloud().tobytes()
    on.set_output_records(True)
    # reset keeps the setting: the replay after it equals a fresh oracle's
    on.reset()
    orc2 = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    for pts, pose in seq[:3]:
        rec, step, offs = make_records(pts, "xyzirt22")
        on.push_raw_cloud_and_pose(rec, pose, point_step=step, offsets=offs)
        orc2.push_raw_cloud_and_pose(rec, pose, point_step=step, offsets=offs)
        orc2.filter_cloud()
        assert on.filter_cloud().tobytes() == expected_records(orc2, rec).tobytes()

    # capacity: n * point_step > 32 B x max_points is an error in record mode on the device paths, fine without it
    small = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=1000)
    n, step = 900, 40  # 36000 B > 32000 B
    rec = np.zeros((n, step), np.uint8)
    rec[:, :12] = np.random.default_rng(0).uniform(-5, 5, (n, 3)).astype(np.float32).view(np.uint8)
    d_in, d_out = _alloc(product, n * step), _alloc(product, n * step)
    try:
        _upload(product, d_in, rec)
        pose = seq[0][1]
        small.push_device(d_in.value, n, pose, step, (0, 4, 8, 12))
        small.filter_device(d_out.value, n)
        small.set_output_records(True)
        with pytest.raises(MorError) as e:
            small.push_device(d_in.value, n, pose, step, (0, 4, 8, 12))
        assert e.value.status == ERR_CAPACITY and b"32 B x max_points" in product.last_error(small.h)
        with pytest.raises(MorError) as e:
            SequenceBatch([small]).step_device([d_in.value], [n], [pose], [d_out.value], step, (0, 4, 8, 12))
        assert e.value.status == ERR_CAPACITY
        # batched handles must agree on the mode
        other = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=1000)
        other.push_device(d_in.value, n, pose, step, (0, 4, 8, 12))
        other.filter_device(d_out.value, n)
        with pytest.raises(MorError) as e:
            SequenceBatch([small, other]).step_device([d_in.value] * 2, [10, 10], [pose] * 2, [d_out.value] * 2, step, (0, 4, 8, 12))
        assert e.value.status == ERR_ARG and b"agree" in product.last_error(small.h)
    finally:
        product.device_free(0, d_in)
        product.device_free(0, d_out)


def test_batched_launch_count(product, cfg_dir):
    cfg = cfg_dir / "MOR_config.txt"
    s = Synth(1, 2)
    hs = [MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=s.max_points) for _ in range(4)]
    a, b = SequenceBatch(hs[:2]), SequenceBatch(hs[2:])
    for h in hs[2:]:
        h.set_output_records(True)
    d_in, d_out = _alloc(product, s.max_points * 32), [_alloc(product, s.max_points * 32) for _ in range(4)]
    try:
        for f in range(3):
            pts, pose = s.frame(f)
            _upload(product, d_in, pts)
            c0 = [hs[0].launch_count(), hs[2].launch_count()]
            a.step_device([d_in.value] * 2, [len(pts)] * 2, [pose] * 2, [d_out[0].value, d_out[1].value])
            b.step_device([d_in.value] * 2, [len(pts)] * 2, [pose] * 2, [d_out[2].value, d_out[3].value])
            assert hs[2].launch_count() - c0[1] == hs[0].launch_count() - c0[0] + 1
            for h in hs:
                h.sync()
    finally:
        for p in [d_in] + d_out:
            product.device_free(0, p)


@pytest.mark.parametrize("stream", [False, True])
def test_harness_keep_fields_writes_the_input_records(built, tmp_path, stream):
    """mov_harness --replay --out with --keep-fields (the C++ class's setKeepInputFields, or the pipelined calls with
    --stream) writes the input's 16-byte records as they are: byte-identical to the PointXYZI run's 32 -> 16 conversion."""
    import subprocess

    from helpers import ROOT
    from test_gpu_harness import _write_replay_dir
    exe = ROOT / "harness" / "mov_harness"
    if not exe.exists():
        subprocess.check_call(["make", "-C", str(ROOT / "harness")])
    s = Synth(1, 1)
    n = 9
    d = tmp_path / "rec"
    _write_replay_dir(d, [s.frame(f) for f in range(n)], 7)
    cfg = ROOT / "config" / "MOR_config.txt"
    outs = {}
    for keep in (False, True):
        o = tmp_path / f"out{int(keep)}"
        o.mkdir()
        cmd = [str(exe), str(cfg), "--replay", str(d), "--out", str(o)] + (["--stream"] if stream else []) + (["--keep-fields"] if keep else [])
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
        assert res.returncode == 0, res.stderr
        outs[keep] = [(o / f"{f:06d}.bin").read_bytes() for f in range(n)]
    assert outs[True] == outs[False]
    assert sum(len(b) for b in outs[True]) > 0
