"""Pipelined against one-kernel-per-frame launches (mor_set_pipelining) for the configurations the pipelined launch variants
serve: the voxel ground modes (k_frame_pipe_ground), method 1 (k_frame_pipe_pde) and both (k_frame_pipe_ground_pde).

For every configuration, two workloads, each with both launch modes alternated round by round in one run (every round
starts from mor_reset, warms up W frames, then times T frames with a host clock that ends in a sync):
  device    push_device + filter_device(None, 0, want_count=False) on 16-byte records staged in HBM, one buffer per frame
  stream    end-to-end submit_frame / collect_frame, 16-byte records in pinned host memory, four frames in flight
Before timing, the last frame's output bytes of the two modes are compared on both paths. One JSON line per configuration
and workload with frames/s per mode (median over the rounds), launches per frame and the GPU's name and power limit
(read-only nvidia-smi query in the same run). --sweep GF,... also times the device path with the front half on GF CTAs
(MOR_PIPE_GF, the launch's tuning override) to choose each variant's CTA split.

    python tools/pipe_modes_run.py [--steps 60] [--warmup 5] [--rounds 5] [--only NAME,...] [--sweep 125,116,107]"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from dynamicslamtool_b200 import MovingObjectRemoval, Synth, load_product  # noqa: E402
from helpers import write_cfg  # noqa: E402

CFG = ROOT / "config"
CONFIGS = {  # name -> (scenario, base config, overrides)
    "c4_ground1": (4, "MOR_config_terrain.txt", {"ground_mode": 1}),
    "c4_ground2": (4, "MOR_config_terrain.txt", {"ground_mode": 2}),
    "c1_method1": (1, "MOR_config.txt", {"method_choice": 1}),
    "hdl64_method1": (2, "MOR_config_hdl64.txt", {"method_choice": 1}),
    "c4_ground2_method1": (4, "MOR_config_terrain.txt", {"ground_mode": 2, "method_choice": 1}),
}


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


def pinned(b, shape):
    nbytes = int(np.prod(shape)) * 4
    p = C.c_void_p()
    assert b.alloc_pinned(nbytes, C.byref(p)) == 0
    return np.frombuffer((C.c_uint8 * nbytes).from_address(p.value), np.float32).reshape(shape)


def device_output(b, h):
    n = h.counts()["NOUT"]
    out = np.empty((n, 8), np.float32)
    if n:
        assert b.device_download(0, out.ctypes.data_as(C.c_void_p), C.c_void_p(h.output_device()), out.nbytes) == 0
    return out


def run_device(h, d_fr, frames, W):
    """All frames; returns (frames/s over frames W.., launches per timed frame)."""
    h.reset()
    for f, (pts, pose) in enumerate(frames):
        if f == W:
            h.sync()
            t0, l0 = time.perf_counter(), h.launch_count()
        h.push_device(d_fr[f], len(pts), pose)
        h.filter_device(None, 0, want_count=False)
    h.sync()
    T = len(frames) - W
    return T / (time.perf_counter() - t0), (h.launch_count() - l0) / T


def run_stream(h, hin, hout, frames, W):
    """All frames through submit / collect; returns (frames/s over frames W.., the last frame's output)."""
    h.reset()
    last = None
    for f, (pts, pose) in enumerate(frames):
        if f == W:
            while h.frames_in_flight():
                h.collect_frame()
            t0 = time.perf_counter()
        if h.frames_in_flight() == 4:
            last = h.collect_frame()
        h.submit_frame(hin[f][: len(pts)], pose, hout[f % 4])
    while h.frames_in_flight():
        last = h.collect_frame()
    return (len(frames) - W) / (time.perf_counter() - t0), last.copy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--only", default="")
    ap.add_argument("--sweep", default="")
    args = ap.parse_args()
    b = load_product()
    name, power = gpu_info()
    W, T = args.warmup, args.steps
    F = W + T
    tmp = Path(tempfile.mkdtemp(prefix="pipe_modes_"))
    sweep = [int(v) for v in args.sweep.split(",") if v]
    for cname, (scenario, base, ov) in CONFIGS.items():
        if args.only and cname not in args.only.split(","):
            continue
        cfg = write_cfg(tmp, name=f"{cname}.txt", base=CFG / base, **ov)
        syn = Synth(scenario, scenario)
        maxp = syn.max_points
        frames = [syn.frame(f) for f in range(F)]
        kw = dict(binding=b, max_points=maxp, max_cells=1 << 21)
        d_fr = [dalloc(b, maxp * 16) for _ in range(F)]
        for f, (pts, _) in enumerate(frames):
            assert b.device_upload(0, C.c_void_p(d_fr[f]), pts.ctypes.data_as(C.c_void_p), pts.nbytes) == 0

        # ---- device-resident
        hs = {m: MovingObjectRemoval(cfg, 4, 3, **kw) for m in (False, True)}
        for m, h in hs.items():
            h.set_pipelining(m)
        run_device(hs[False], d_fr, frames, W)
        run_device(hs[True], d_fr, frames, W)
        same = device_output(b, hs[False]).tobytes() == device_output(b, hs[True]).tobytes()
        assert same, f"{cname}: the last frame's output differs between the launch modes (device path)"
        res = {False: [], True: []}
        launches = {}
        for _ in range(args.rounds):
            for m, h in hs.items():
                fps, lpf = run_device(h, d_fr, frames, W)
                res[m].append(fps)
                launches[m] = lpf
        print(json.dumps({"config": cname, "workload": "device", "gpu": name, "power_limit": power, "frames": T, "rounds": args.rounds,
                          "pipelined_fps": round(statistics.median(res[True]), 1), "unpipelined_fps": round(statistics.median(res[False]), 1),
                          "pipelined_fps_all": [round(v, 1) for v in res[True]], "unpipelined_fps_all": [round(v, 1) for v in res[False]],
                          "launches_per_frame": {"pipelined": launches[True], "unpipelined": launches[False]}}), flush=True)
        if sweep:
            res = {gf: [] for gf in sweep}
            for _ in range(args.rounds):
                for gf in sweep:
                    os.environ["MOR_PIPE_GF"] = str(gf)
                    res[gf].append(run_device(hs[True], d_fr, frames, W)[0])
            os.environ.pop("MOR_PIPE_GF", None)
            print(json.dumps({"config": cname, "workload": "device_split_sweep", "gpu": name, "power_limit": power,
                              "front_ctas_fps": {gf: round(statistics.median(v), 1) for gf, v in res.items()}}), flush=True)
        for h in hs.values():
            h.close()

        # ---- streaming end to end
        hin = [pinned(b, (maxp, 4)) for _ in range(F)]
        for f, (pts, _) in enumerate(frames):
            hin[f][: len(pts)] = pts
        hout = {m: [pinned(b, (maxp, 8)) for _ in range(4)] for m in (False, True)}
        hs = {m: MovingObjectRemoval(cfg, 4, 3, **kw) for m in (False, True)}
        for m, h in hs.items():
            h.set_pipelining(m)
        outs = {m: run_stream(h, hin, hout[m], frames, W)[1] for m, h in hs.items()}
        assert outs[False].tobytes() == outs[True].tobytes(), f"{cname}: the last frame's output differs between the launch modes (stream path)"
        res = {False: [], True: []}
        for _ in range(args.rounds):
            for m, h in hs.items():
                res[m].append(run_stream(h, hin, hout[m], frames, W)[0])
        print(json.dumps({"config": cname, "workload": "stream", "gpu": name, "power_limit": power, "frames": T, "rounds": args.rounds,
                          "pipelined_fps": round(statistics.median(res[True]), 1), "unpipelined_fps": round(statistics.median(res[False]), 1),
                          "pipelined_fps_all": [round(v, 1) for v in res[True]], "unpipelined_fps_all": [round(v, 1) for v in res[False]]}),
              flush=True)
        for h in hs.values():
            h.close()
        for d in d_fr:
            b.device_free(0, C.c_void_p(d))


if __name__ == "__main__":
    main()
