"""Quick device-resident timing of one build on the C2 sequence (not the bench: no clocks check, no e2e).
usage: [MOR_PRODUCT_LIB=...] [QB_PIPE=1] python tools/quick_bench.py [frames=120] [warmup=20]
Prints frames/s, the mean in-kernel phase times and a crc of the last output (equal across correct builds).
QB_PIPE=1: pipelined launches, and instead of the one-kernel-per-frame phases the mean timeline of each half of a fused
launch (front half of frame f+1 beside the back half of f; the TS_FRONT / TS_BACK words of phase_ts)."""
import ctypes as C, sys, zlib, numpy as np
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from dynamicslamtool_b200 import MovingObjectRemoval, Synth, load_product
F = int(sys.argv[1]) if len(sys.argv) > 1 else 120
W = int(sys.argv[2]) if len(sys.argv) > 2 else 20
import os
STEP = int(os.environ.get("QB_STEP", "16"))  # 22: the velodyne XYZIRT record (x, y, z, intensity, ring u16, time f32), unaligned
b = load_product()
s = Synth(2, 2)
maxp = s.max_points
frames = [s.frame(f) for f in range(F)]
def pack(pts):
    if STEP == 16: return pts
    rec = np.zeros((len(pts), STEP), np.uint8)
    rec[:, :16] = pts.view(np.uint8).reshape(len(pts), 16)
    return rec
d = C.c_void_p()
SLOT = maxp * 32
assert b.device_alloc(0, F * SLOT, C.byref(d)) == 0
for f, (pts, _) in enumerate(frames):
    rec = pack(pts)
    assert b.device_upload(0, C.c_void_p(d.value + f * SLOT), rec.ctypes.data_as(C.c_void_p), rec.nbytes) == 0
m = MovingObjectRemoval('config/MOR_config_hdl64.txt', 4, 3, binding=b, max_points=maxp)
if os.environ.get("QB_PIPE"): m.set_pipelining(True)
for rep in range(2):  # second pass timed (first warms everything incl. clocks)
    m.reset()
    for f in range(W):
        m.push_device(d.value + f * SLOT, len(frames[f][0]), frames[f][1], point_step=STEP); m.filter_device(None, 0, want_count=False)
    m.sync(); m.event_record(0)
    for f in range(W, F):
        m.push_device(d.value + f * SLOT, len(frames[f][0]), frames[f][1], point_step=STEP); m.filter_device(None, 0, want_count=False)
    m.event_record(1)
    ms = m.event_elapsed_ms(0, 1)
c = m.counts()
out = np.empty((c["NOUT"], 8), np.float32)
b.device_download(0, out.ctypes.data_as(C.c_void_p), C.c_void_p(m.output_device()), out.nbytes)
print(f"{(F - W) / (ms * 1e-3):8.0f} frames/s  {1e3 * ms / (F - W):7.1f} us/frame  crc {zlib.crc32(out.tobytes()):08x} errflags {c['ERRFLAGS']}")
if os.environ.get("QB_PIPE"):
    # per-half timeline of the fused launches (CTA 0 of each half at its barriers, the last CTA out at the end), in us,
    # averaged over the frames after the warm-up, with a sync per frame
    TS_FRONT, TS_BACK = 12, 21
    FRONT = ["ingest", "cells", "link", "test", "jump", "cross", "roots+select", "end"]
    BACK = ["housekeeping", "stats+transform+match", "moving+chain", "filter"]
    ts = (C.c_ulonglong * 32)()
    m.reset()
    acc = np.zeros(len(FRONT) + len(BACK))
    n = 0
    for f in range(F):
        m.push_device(d.value + f * SLOT, len(frames[f][0]), frames[f][1], point_step=STEP)
        if f > W:  # (this push launched the front half of f beside the back half of f - 1)
            assert b.lib.mor_debug_phase_ts(m.h, ts) == 0
            w = np.array(ts[:], np.float64)
            fr = np.diff(w[TS_FRONT:TS_FRONT + len(FRONT) + 1])
            bk = np.diff(w[TS_BACK:TS_BACK + len(BACK) + 1])
            acc += np.concatenate([fr, bk]) * 1e-3
            n += 1
        m.filter_device(None, 0, want_count=False)
    acc /= max(n, 1)
    print("  front " + "  ".join(f"{k} {v:.1f}" for k, v in zip(FRONT, acc[:len(FRONT)])) + f"  total {acc[:len(FRONT)].sum():.1f}")
    print("  back  " + "  ".join(f"{k} {v:.1f}" for k, v in zip(BACK, acc[len(FRONT):])) + f"  total {acc[len(FRONT):].sum():.1f}")
    sys.exit(0)
# phase timeline, averaged over a second pass with a sync per frame
m.reset()
acc = {}
for f in range(F):
    m.push_device(d.value + f * SLOT, len(frames[f][0]), frames[f][1], point_step=STEP); m.filter_device(None, 0, want_count=True)
    if f >= W:
        for k, v in m.phase_times().items(): acc[k] = acc.get(k, 0.0) + v
print("  " + "  ".join(f"{k[3:]} {v / (F - W):.1f}" for k, v in acc.items()), " sum %.1f" % (sum(acc.values()) / (F - W)))
