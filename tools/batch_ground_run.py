"""Batched against sequential stepping of the voxel ground mode (BASELINE config C4: MOR_config_terrain.txt, ground_mode 2).

For every S, the same S handles (distinct seeds of Synth(4, .), frames staged in HBM beforehand) run two arms, each from a
fresh state (mor_reset) with 3 warm-up steps and then T timed steps:
  batched     SequenceBatch.step_device: 9 ground launches + 1 frame launch per step for all S sequences
  sequential  every handle in turn: push_device + filter_device(d_out, cap, want_count=False)
A host clock times the T steps and ends with a sync of every handle. One JSON line per S: frames/s of each arm, kernel
launches per step (launch_count()), whether the last step's outputs of the two arms are byte-equal per sequence, and the
GPU's name and power limit (read-only nvidia-smi query in the same run).

    python tools/batch_ground_run.py [--S 1 8 16 37] [--steps 40]"""
import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from dynamicslamtool_b200 import MovingObjectRemoval, SequenceBatch, Synth, load_product  # noqa: E402

CFG = ROOT / "config" / "MOR_config_terrain.txt"


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip()
        name, power = [v.strip() for v in out.split(",", 1)]
        return name, power
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--S", type=int, nargs="+", default=[1, 8, 16, 37])
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    b = load_product()
    Smax, W, T = max(args.S), args.warmup, args.steps
    F = W + T
    syn = [Synth(4, 1000 + s) for s in range(Smax)]
    maxp = syn[0].max_points
    # frames staged in HBM: d_frames[s][f], n[s][f], pose[s][f]
    d_frames, ns, poses = [], [], []
    for s in range(Smax):
        row, rn, rp = [], [], []
        for f in range(F):
            pts, pose = syn[s].frame(f)
            p = C.c_void_p()
            assert b.device_alloc(0, max(pts.nbytes, 16), C.byref(p)) == 0
            assert b.device_upload(0, p, pts.ctypes.data_as(C.c_void_p), pts.nbytes) == 0
            row.append(p.value); rn.append(pts.shape[0]); rp.append(pose)
        d_frames.append(row); ns.append(rn); poses.append(rp)
    d_out = {}
    for arm in ("batched", "sequential"):
        d_out[arm] = []
        for _ in range(Smax):
            p = C.c_void_p()
            assert b.device_alloc(0, maxp * 32, C.byref(p)) == 0
            d_out[arm].append(p.value)
    name, power = gpu_info()
    for S in args.S:
        hs = [MovingObjectRemoval(CFG, 4, 3, binding=b, max_points=maxp, max_cells=1 << 21) for _ in range(S)]
        batch = SequenceBatch(hs)
        res = {"workload": "C4 batched vs sequential", "S": S, "steps": T, "warmup": W, "gpu": name, "power_limit": power}
        outs = {}
        for arm in ("batched", "sequential"):
            for h in hs:
                h.reset()

            def step(f, arm=arm):
                if arm == "batched":
                    batch.step_device([d_frames[s][f] for s in range(S)], [ns[s][f] for s in range(S)], [poses[s][f] for s in range(S)],
                                      d_out[arm][:S])
                else:
                    for s, h in enumerate(hs):
                        h.push_device(d_frames[s][f], ns[s][f], poses[s][f])
                        h.filter_device(d_out[arm][s], maxp, want_count=False)

            for f in range(W):
                step(f)
            for h in hs:
                h.sync()
            l0 = sum(h.launch_count() for h in hs)
            t0 = time.perf_counter()
            for f in range(W, F):
                step(f)
            for h in hs:
                h.sync()
            dt = time.perf_counter() - t0
            res[f"{arm}_frames_per_s"] = round(S * T / dt, 1)
            res[f"{arm}_launches_per_step"] = (sum(h.launch_count() for h in hs) - l0) / T
            o = []
            for s, h in enumerate(hs):
                n = h.counts()["NOUT"]
                buf = np.empty((n, 8), np.float32)
                if n:
                    assert b.device_download(0, buf.ctypes.data_as(C.c_void_p), C.c_void_p(d_out[arm][s]), n * 32) == 0
                o.append(buf.tobytes())
            outs[arm] = o
        res["speedup"] = round(res["batched_frames_per_s"] / res["sequential_frames_per_s"], 3)
        res["outputs_equal_per_sequence"] = [a == c for a, c in zip(outs["batched"], outs["sequential"])]
        res["outputs_equal"] = all(res["outputs_equal_per_sequence"])
        print(json.dumps(res), flush=True)
        for h in hs:
            h.close()
    for row in d_frames:
        for p in row:
            b.device_free(0, C.c_void_p(p))
    for arm in d_out:
        for p in d_out[arm]:
            b.device_free(0, C.c_void_p(p))


if __name__ == "__main__":
    main()
