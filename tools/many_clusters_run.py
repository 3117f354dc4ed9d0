"""Frames with many clusters: frames/s and the frame kernel's phase times (mor_get_phase_times) at K ~ 8k (the single-CTA
steps), 16k (their last size), 16,385 and 30k and 100k (the group-wide steps of the large-K path), device-resident, with and
without pipelined launches (alternated round by round in one run).

The scene is tests/test_gpu_many_clusters.py's: a lattice of isolated points, one cluster each at min_cluster_size 1, plus
four moving blobs (the static points are reciprocal matches of themselves every frame; the blobs are matched, flagged and
removed). Every round starts from mor_reset, runs W frames, then times T frames with a host clock that ends in a sync.
The phase times are those of the last frame of a round without pipelining (one kernel per frame). The frames repeat the
scene's FRAMES-frame cycle. One JSON line per K with the GPU's name and power limit (read-only nvidia-smi query in the
same run).

    python tools/many_clusters_run.py [--steps 20] [--warmup 4] [--rounds 3] [--only 8k,16k,...]"""
import argparse
import ctypes as C
import json
import statistics
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))
from dynamicslamtool_b200 import MovingObjectRemoval, load_product  # noqa: E402
from helpers import IDENTITY_POSE  # noqa: E402
from pipe_modes_run import dalloc, gpu_info  # noqa: E402
from test_gpu_many_clusters import MAX_CLUSTERS, N_BAD, N_GOOD, scene_cfg, scene_frames  # noqa: E402

SIZES = {"8k": 8_000, "16k": 16_384, "16385": 16_385, "30k": 30_000, "100k": 100_000}


def run_round(h, d, ns, W, T, pipelining):
    h.reset()
    h.set_pipelining(pipelining)
    for f in range(W + T):
        if f == W:
            h.sync()
            t0 = time.perf_counter()
        h.push_device(d[f % len(d)], ns[f % len(d)], IDENTITY_POSE)
        h.filter_device(None, 0, want_count=False)
    h.sync()
    h.counts()  # (runs a pending back half)
    return T / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    name, power = gpu_info()
    b = load_product()
    cfg = scene_cfg(tempfile.mkdtemp())
    for tag, k in SIZES.items():
        if args.only and tag not in args.only.split(","):
            continue
        frames = scene_frames(k)
        maxp = max(len(p) for p in frames)
        d = []
        for pts in frames:
            d.append(dalloc(b, pts.nbytes))
            assert b.device_upload(0, C.c_void_p(d[-1]), pts.ctypes.data_as(C.c_void_p), pts.nbytes) == 0
        ns = [len(p) for p in frames]
        h = MovingObjectRemoval(cfg, N_BAD, N_GOOD, binding=b, max_points=maxp, max_clusters=MAX_CLUSTERS)
        fps = {"plain": [], "pipelined": []}
        phases = None
        for _ in range(args.rounds):
            fps["plain"].append(run_round(h, d, ns, args.warmup, args.steps, False))
            phases = h.phase_times()
            fps["pipelined"].append(run_round(h, d, ns, args.warmup, args.steps, True))
        c = h.counts()
        print(json.dumps({"K": tag, "clusters": c["K"], "points": ns[0], "errflags": c["ERRFLAGS"],
                          "fps_plain": round(statistics.median(fps["plain"]), 1), "fps_pipelined": round(statistics.median(fps["pipelined"]), 1),
                          "fps_rounds": {m: [round(v, 1) for v in vs] for m, vs in fps.items()},
                          "phase_us": {p: round(v, 1) for p, v in phases.items()}, "gpu": name, "power_limit": power}), flush=True)
        h.close()
        for p in d:
            b.device_free(0, C.c_void_p(p))


if __name__ == "__main__":
    main()
