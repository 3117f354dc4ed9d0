"""A fleet of LiDAR recordings of different sensors and lengths on one GPU, three ways (BASELINE.md, mixed batched steps):

  1. mixed: mor_batch_step_device_mixed over `--slots` slots; a slot takes the next recording (mor_reset of a handle
     with that recording's config) as soon as its current one ends;
  2. lockstep: the best mor_batch_step_device allows. The recordings of one config in batches of up to `--slots`; a
     batch steps until its longest recording ends, finished sequences are dropped from it;
  3. alone: every recording on a handle of its own, push_device + filter_device frame by frame.

    python tools/mixed_batch_run.py [--slots 37] [--recordings 111] [--seed 0] [--repeats 3]

Recordings: C1, C2 or C3 (Synth(1|2|3, seed) with its config), 8 to 64 frames, drawn with the seed; the frames come from
four generated streams per config, staged in HBM before anything is timed. Before timing, the last frame of every
recording is compared byte for byte between ways 1 and 3. Timed: host clock from the first step to the device
synchronisation after the last, the three ways alternating `--repeats` times. Prints one JSON line per way and repeat
and a summary line with the card's name and power limit.
"""
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
from dynamicslamtool_b200 import MixedBatch, MovingObjectRemoval, SequenceBatch, Synth, load_product  # noqa: E402

CONFIGS = {1: "MOR_config.txt", 2: "MOR_config_hdl64.txt", 3: "MOR_config_os128.txt"}
STREAMS, MAX_LEN = 4, 64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slots", type=int, default=37)
    ap.add_argument("--recordings", type=int, default=111)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    b = load_product()
    rng = np.random.default_rng(args.seed)
    recs = [(int(rng.integers(1, 4)), int(rng.integers(0, STREAMS)), int(rng.integers(8, MAX_LEN + 1))) for _ in range(args.recordings)]
    # staged frames: [config][stream][frame] -> (device address, n, pose)
    maxp = {sc: Synth(sc, 0).max_points for sc in CONFIGS}
    staged, bufs = {}, []
    for sc in CONFIGS:
        for k in range(STREAMS):
            syn = Synth(sc, 100 * sc + k)
            frames = [syn.frame(f) for f in range(MAX_LEN)]
            d = C.c_void_p()
            assert b.device_alloc(0, MAX_LEN * maxp[sc] * 16, C.byref(d)) == 0
            bufs.append(d)
            for f, (pts, pose) in enumerate(frames):
                assert b.device_upload(0, C.c_void_p(d.value + f * maxp[sc] * 16), pts.ctypes.data_as(C.c_void_p), pts.nbytes) == 0
                staged[(sc, k, f)] = (d.value + f * maxp[sc] * 16, len(pts), pose)
    total_frames = sum(r[2] for r in recs)

    def out_buf(sc):
        d = C.c_void_p()
        assert b.device_alloc(0, maxp[sc] * 32, C.byref(d)) == 0
        bufs.append(d)
        return d.value

    make = lambda sc: MovingObjectRemoval(ROOT / "config" / CONFIGS[sc], 4, 3, binding=b, max_points=maxp[sc])  # noqa: E731
    # way 1: per slot one handle of each config and one output buffer of the largest size
    slots = [{sc: make(sc) for sc in CONFIGS} for _ in range(args.slots)]
    slot_out = [out_buf(3) for _ in range(args.slots)]
    mixed = MixedBatch(b)

    def last_output(h, d_out):
        h.sync()
        n = h.counts()["NOUT"]
        out = np.empty(n * 32, np.uint8)
        if n:
            assert b.device_download(0, out.ctypes.data_as(C.c_void_p), C.c_void_p(d_out), out.nbytes) == 0
        return out

    def run_mixed(keep_last=False):
        queue = list(range(len(recs)))
        cur = [None] * args.slots  # (recording, next frame)
        last, steps, launches0 = {}, 0, sum(h.launch_count() for s in slots for h in s.values())
        while True:
            for i in range(args.slots):
                if cur[i] is None and queue:
                    r = queue.pop(0)
                    slots[i][recs[r][0]].reset()
                    cur[i] = (r, 0)
            active = [i for i in range(args.slots) if cur[i] is not None]
            if not active:
                break
            hs, ptrs, ns, poses, outs = [], [], [], [], []
            for i in active:
                r, f = cur[i]
                sc, k, _ = recs[r]
                d, n, pose = staged[(sc, k, f)]
                hs.append(slots[i][sc]); ptrs.append(d); ns.append(n); poses.append(pose); outs.append(slot_out[i])
            mixed.step(hs, ptrs, ns, poses, outs)
            steps += 1
            for i in active:
                r, f = cur[i]
                if f + 1 == recs[r][2]:
                    if keep_last:
                        last[r] = last_output(slots[i][recs[r][0]], slot_out[i])
                    cur[i] = None
                else:
                    cur[i] = (r, f + 1)
        for s in slots:
            for h in s.values():
                h.sync()
        return last, steps, sum(h.launch_count() for s in slots for h in s.values()) - launches0

    # way 2: per config `slots` handles, batches of the recordings of that config
    lock = {sc: [make(sc) for _ in range(args.slots)] for sc in CONFIGS}
    lock_out = {sc: [out_buf(sc) for _ in range(args.slots)] for sc in CONFIGS}

    def run_lockstep():
        steps, launches0 = 0, sum(h.launch_count() for hs in lock.values() for h in hs)
        for sc in CONFIGS:
            mine = [r for r in range(len(recs)) if recs[r][0] == sc]
            for c in range(0, len(mine), args.slots):
                group = mine[c:c + args.slots]
                for j in range(len(group)):
                    lock[sc][j].reset()
                for f in range(max(recs[r][2] for r in group)):
                    live = [j for j, r in enumerate(group) if f < recs[r][2]]
                    batch = SequenceBatch([lock[sc][j] for j in live])
                    fr = [staged[(sc, recs[group[j]][1], f)] for j in live]
                    batch.step_device([x[0] for x in fr], [x[1] for x in fr], [x[2] for x in fr], [lock_out[sc][j] for j in live])
                    steps += 1
        for hs in lock.values():
            for h in hs:
                h.sync()
        return steps, sum(h.launch_count() for hs in lock.values() for h in hs) - launches0

    # way 3: one handle per config, every recording alone
    alone = {sc: make(sc) for sc in CONFIGS}
    alone_out = {sc: out_buf(sc) for sc in CONFIGS}

    def run_alone(keep_last=False):
        last, launches0 = {}, sum(h.launch_count() for h in alone.values())
        for r, (sc, k, length) in enumerate(recs):
            h = alone[sc]
            h.reset()
            for f in range(length):
                d, n, pose = staged[(sc, k, f)]
                h.push_device(d, n, pose)
                h.filter_device(alone_out[sc], maxp[sc], want_count=False)
            if keep_last:
                last[r] = last_output(h, alone_out[sc])
        for h in alone.values():
            h.sync()
        return last, total_frames, sum(h.launch_count() for h in alone.values()) - launches0

    # outputs first: the last frame of every recording, mixed against alone
    got, _, _ = run_mixed(keep_last=True)
    want, _, _ = run_alone(keep_last=True)
    bad = [r for r in range(len(recs)) if got[r].tobytes() != want[r].tobytes()]
    if bad:
        raise SystemExit(f"mixed and alone outputs differ in recordings {bad[:10]}")
    run_lockstep()  # warm-up of the third way
    gpu = card()
    rows = {"mixed": [], "lockstep": [], "alone": []}
    for rep in range(args.repeats):
        for way in ("mixed", "lockstep", "alone"):
            t0 = time.perf_counter()
            if way == "mixed":
                _, steps, launches = run_mixed()
            elif way == "lockstep":
                steps, launches = run_lockstep()
            else:
                _, steps, launches = run_alone()
            dt = time.perf_counter() - t0
            row = {"way": way, "repeat": rep, "frames": total_frames, "seconds": round(dt, 4), "frames_per_s": round(total_frames / dt, 1),
                   "steps": steps, "launches_per_step": round(launches / steps, 2)}
            rows[way].append(row)
            print(json.dumps(row), flush=True)
    counts = {f"C{sc}": sum(1 for r in recs if r[0] == sc) for sc in CONFIGS}
    print(json.dumps({"summary": {w: [r["frames_per_s"] for r in v] for w, v in rows.items()}, "gpu": gpu, "slots": args.slots,
                      "recordings": counts, "frames": total_frames, "outputs_checked": len(recs)}), flush=True)
    for d in bufs:
        b.device_free(0, d)


if __name__ == "__main__":
    main()
