"""PointXYZI output against output records (mor_set_output_records) on C2 (Synth(2, .), MOR_config_hdl64.txt).

Three workloads, each with both output modes alternated round by round in one run (every round starts from mor_reset,
warms up W frames, then times T frames with a host clock that ends in a sync):
  device    device-resident pipelined push_device + filter_device(None, 0, want_count=False); input 22-byte XYZIRT records
            staged in HBM; output records are 22 B, PointXYZI records 32 B
  stream    end-to-end submit_frame / collect_frame with pipelining, 16-byte records in pinned host memory: the D2H copy of
            output records is half that of PointXYZI records
  batch     SequenceBatch.step_device with S = 37 sequences (4 distinct seeds), 22-byte records
Before timing, every frame of the device and stream workloads is checked in record mode against the records the CPU
oracle's bookkeeping selects (tests/records_ref.py). One JSON line per workload with frames/s per mode (median over the
rounds), launches per frame and the GPU's name and power limit (read-only nvidia-smi query in the same run).

    python tools/records_run.py [--steps 60] [--warmup 5] [--rounds 5] [--check-frames 12]"""
import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from dynamicslamtool_b200 import MorBinding, MovingObjectRemoval, SequenceBatch, Synth, load_product  # noqa: E402
from records_ref import LAYOUTS, expected_records, make_records  # noqa: E402

CFG = ROOT / "config" / "MOR_config_hdl64.txt"


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip()
        name, power = [v.strip() for v in out.split(",", 1)]
        return name, power
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def dalloc(b, nbytes):
    p = C.c_void_p()
    assert b.device_alloc(0, max(nbytes, 16), C.byref(p)) == 0
    return p.value


def upload(b, d, a):
    if a.nbytes:
        assert b.device_upload(0, C.c_void_p(d), a.ctypes.data_as(C.c_void_p), a.nbytes) == 0


def download(b, d, n, step):
    out = np.empty((n, step), np.uint8)
    if n:
        assert b.device_download(0, out.ctypes.data_as(C.c_void_p), C.c_void_p(d), n * step) == 0
    return out


def pinned(b, shape):
    nbytes = int(np.prod(shape))
    p = C.c_void_p()
    assert b.alloc_pinned(nbytes, C.byref(p)) == 0
    return np.frombuffer((C.c_uint8 * nbytes).from_address(p.value), np.uint8).reshape(shape), p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--check-frames", type=int, default=12)
    ap.add_argument("--S", type=int, default=37)
    args = ap.parse_args()
    b = load_product()
    orc_b = MorBinding(C.CDLL(str(ROOT / "oracle" / "libmor_oracle.so")), "oracle_")
    name, power = gpu_info()
    W, T = args.warmup, args.steps
    F = W + T
    syn = Synth(2, 2)
    maxp = syn.max_points
    frames = [syn.frame(f) for f in range(F)]
    r22 = [make_records(p, "xyzirt22") for p, _ in frames]
    r16 = [make_records(p, "xyzi16") for p, _ in frames]
    poses = [pose for _, pose in frames]

    # ---- check: record mode equals the oracle-derived records on the first check-frames frames (device and stream paths)
    orc = MovingObjectRemoval(CFG, 4, 3, binding=orc_b)
    m = MovingObjectRemoval(CFG, 4, 3, binding=b, max_points=maxp)
    m.set_output_records(True)
    m.set_pipelining(True)
    d_chk, d_out = dalloc(b, maxp * 32), dalloc(b, maxp * 32)
    want16 = []
    for f in range(args.check_frames):
        rec, step, offs = r22[f]
        orc.push_raw_cloud_and_pose(rec, poses[f], point_step=step, offsets=offs)
        orc.filter_cloud()
        upload(b, d_chk, rec)
        m.push_device(d_chk, len(rec), poses[f], step, offs)
        n = m.filter_device(d_out, maxp)
        m.sync()  # (the device-to-device copy runs on the handle's stream)
        assert download(b, d_out, n, step).tobytes() == expected_records(orc, rec).tobytes(), f"device path: frame {f} differs from the oracle"
        want16.append(expected_records(orc, r16[f][0]).tobytes())
    ms = MovingObjectRemoval(CFG, 4, 3, binding=b, max_points=maxp)
    ms.set_output_records(True)
    ms.set_pipelining(True)
    ins = [pinned(b, (maxp, 16)) for _ in range(4)]
    outs = [pinned(b, (maxp, 16)) for _ in range(4)]
    got = []
    for f in range(args.check_frames):
        rec, step, offs = r16[f]
        ins[f % 4][0][: len(rec)] = rec
        ms.submit_frame(ins[f % 4][0][: len(rec)], poses[f], outs[f % 4][0], point_step=step, offsets=offs)
        if f >= 3:
            got.append(ms.collect_frame().tobytes())
    while ms.frames_in_flight():
        got.append(ms.collect_frame().tobytes())
    assert got == want16, "stream path differs from the oracle"
    ms.close()
    print(json.dumps({"check": "ok", "frames": args.check_frames}), flush=True)

    # ---- device-resident pipelined, 22-byte input records staged in HBM
    step22, offs22 = 22, LAYOUTS["xyzirt22"][1]
    d_fr = [dalloc(b, maxp * step22) for _ in range(F)]
    for f in range(F):
        upload(b, d_fr[f], r22[f][0])
    hs = {False: MovingObjectRemoval(CFG, 4, 3, binding=b, max_points=maxp), True: m}
    for rec_mode, h in hs.items():
        h.set_output_records(rec_mode)
        h.set_pipelining(True)
    res = {False: [], True: []}
    launches = {}
    for _ in range(args.rounds):
        for rec_mode, h in hs.items():
            h.reset()
            for f in range(F):
                if f == W:
                    h.sync()
                    t0, l0 = time.perf_counter(), h.launch_count()
                h.push_device(d_fr[f], len(r22[f][0]), poses[f], step22, offs22)
                h.filter_device(None, 0, want_count=False)
            h.sync()
            res[rec_mode].append(T / (time.perf_counter() - t0))
            launches[rec_mode] = (h.launch_count() - l0) / T
    print(json.dumps({"workload": "device_pipelined_c2_xyzirt22", "gpu": name, "power_limit": power, "frames": T, "rounds": args.rounds,
                      "xyzi_fps": round(statistics.median(res[False]), 1), "records_fps": round(statistics.median(res[True]), 1),
                      "xyzi_fps_all": [round(v, 1) for v in res[False]], "records_fps_all": [round(v, 1) for v in res[True]],
                      "launches_per_frame": {"xyzi": launches[False], "records": launches[True]}}), flush=True)

    # ---- streaming end to end, 16-byte records from pinned host memory
    hin = [pinned(b, (maxp, 16)) for _ in range(F)]
    for f in range(F):
        hin[f][0][: len(r16[f][0])] = r16[f][0]
    hout = {False: [pinned(b, (maxp, 32)) for _ in range(4)], True: [pinned(b, (maxp, 16)) for _ in range(4)]}
    sh = {False: MovingObjectRemoval(CFG, 4, 3, binding=b, max_points=maxp), True: MovingObjectRemoval(CFG, 4, 3, binding=b, max_points=maxp)}
    res = {False: [], True: []}
    d2h = {False: 0, True: 0}
    for rec_mode, h in sh.items():
        h.set_output_records(rec_mode)
        h.set_pipelining(True)
    for _ in range(args.rounds):
        for rec_mode, h in sh.items():
            h.reset()
            nbytes = 0
            for f in range(F):
                if f == W:
                    while h.frames_in_flight():
                        h.collect_frame()
                    t0, nbytes = time.perf_counter(), 0
                n = len(r16[f][0])
                o = hout[rec_mode][f % 4][0]
                out = o if rec_mode else o.view(np.float32).reshape(maxp, 8)
                if h.frames_in_flight() == 4:
                    nbytes += h.collect_frame().nbytes
                h.submit_frame(hin[f][0][:n], poses[f], out, point_step=16, offsets=(0, 4, 8, 12))
            while h.frames_in_flight():
                nbytes += h.collect_frame().nbytes
            res[rec_mode].append(T / (time.perf_counter() - t0))
            d2h[rec_mode] = nbytes / T
    print(json.dumps({"workload": "stream_e2e_c2_xyzi16", "gpu": name, "power_limit": power, "frames": T, "rounds": args.rounds,
                      "xyzi_fps": round(statistics.median(res[False]), 1), "records_fps": round(statistics.median(res[True]), 1),
                      "xyzi_fps_all": [round(v, 1) for v in res[False]], "records_fps_all": [round(v, 1) for v in res[True]],
                      "d2h_bytes_per_frame": {"xyzi": round(d2h[False]), "records": round(d2h[True])}}), flush=True)

    # ---- batched, S sequences of 22-byte records (4 distinct seeds)
    S, Tb = args.S, max(T // 2, 10)
    Fb = W + Tb
    seeds = [Synth(2, 10 + k) for k in range(4)]
    bseq = [[seeds[k].frame(f) for f in range(Fb)] for k in range(4)]
    bfr = [[make_records(p, "xyzirt22")[0] for p, _ in bseq[k]] for k in range(4)]
    bpose = [[pose for _, pose in bseq[k]] for k in range(4)]
    d_b = [[dalloc(b, maxp * step22) for _ in range(Fb)] for _ in range(4)]
    for k in range(4):
        for f in range(Fb):
            upload(b, d_b[k][f], bfr[k][f])
    d_outs = [dalloc(b, maxp * 32) for _ in range(S)]
    groups = {rm: [MovingObjectRemoval(CFG, 4, 3, binding=b, max_points=maxp) for _ in range(S)] for rm in (False, True)}
    for rm, g in groups.items():
        for h in g:
            h.set_output_records(rm)
    batches = {rm: SequenceBatch(g) for rm, g in groups.items()}
    res = {False: [], True: []}
    launches = {}
    for _ in range(args.rounds):
        for rm, g in groups.items():
            for h in g:
                h.reset()
            for f in range(Fb):
                if f == W:
                    for h in g:
                        h.sync()
                    t0, l0 = time.perf_counter(), g[0].launch_count()
                batches[rm].step_device([d_b[s % 4][f] for s in range(S)], [len(bfr[s % 4][f]) for s in range(S)],
                                        [bpose[s % 4][f] for s in range(S)], d_outs, step22, offs22)
            for h in g:
                h.sync()
            res[rm].append(S * Tb / (time.perf_counter() - t0))
            launches[rm] = (g[0].launch_count() - l0) / Tb
    print(json.dumps({"workload": f"batch_c2_xyzirt22_S{S}", "gpu": name, "power_limit": power, "steps": Tb, "rounds": args.rounds,
                      "xyzi_fps": round(statistics.median(res[False]), 1), "records_fps": round(statistics.median(res[True]), 1),
                      "xyzi_fps_all": [round(v, 1) for v in res[False]], "records_fps_all": [round(v, 1) for v in res[True]],
                      "launches_per_step": {"xyzi": launches[False], "records": launches[True]}}), flush=True)


if __name__ == "__main__":
    main()
