#!/usr/bin/env python
"""bench.py — MOR per-frame filtering hot path on B200 (BASELINE.json metric).

A "step" is one frame through pushRawCloudAndPose + filterCloud. Workload at every N: config C2 of
BASELINE.json — a seeded synthetic HDL-64E street sequence (~130k returns/frame, 5 moving boxes,
config/MOR_config_hdl64.txt); each rank runs its own independent sequence (seed 2 + rank), no
collective on the data path (frames of one sequence are strictly sequential: "replicas only").

  value     frames/s with every input frame already resident in HBM and the output left in HBM
            (mor_push_raw_cloud_and_pose_device / mor_filter_cloud_device, no host sync in the loop)
  e2e       frames/s through the host C ABI: pinned host input, H2D inside push, D2H of the filtered
            cloud inside filter, one stream synchronisation per frame (what a ROS callback would see)
  roofline  the dominant kernel (by summed CUDA-event time) against the measured HBM peak
  cpu_baseline / --impl reference   the CPU oracle (PCL-semantics restatement; the reference itself
            cannot be built offline) on the box's host cores

Timing: CUDA events on the handle's own stream (mor_event_record), max over ranks.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

from dynamicslamtool_b200 import MorBinding, MovingObjectRemoval, Synth, load_product  # noqa: E402

CFG = ROOT / "config" / "MOR_config_hdl64.txt"
SCENARIO = 2
METRIC = "frames/s, pushRawCloudAndPose+filterCloud, 120k-pt HDL-64E frame pairs"
WORKLOAD = "C2: synthetic HDL-64E street sequence (64x2083 rays, ~130k returns/frame, 5 moving boxes), MOR_config_hdl64.txt"


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        self.device, self.samples, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([t.strip() for t in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples if len(s) >= 6 for i in range(4) if s[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def pinned_array(binding: MorBinding, shape, dtype):
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    if binding.alloc_pinned(n, C.byref(p)):
        raise MemoryError("cudaMallocHost failed")
    buf = (C.c_uint8 * n).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape), p


def generate_frames(seed, n_frames, pts_out, counts_out, poses_out):
    s = Synth(SCENARIO, seed)
    for f in range(n_frames):
        pts, pose = s.frame(f, out=pts_out[f])
        counts_out[f] = pts.shape[0]
        poses_out[f] = pose


def algorithmic_bytes(c):
    """SURVEY §8(d) per-frame algorithmic bytes from the logged counts."""
    return (16 * c["N"] + 17 * c["NT"] + 104 * c["NC"] + 24 * c["NKPREV"] + 32 * (c["P1"] + c["P2"]) + 20 * c["NT"] + 16 * c["NOUT"])


def _oracle_worker(orc, frames, maxp, steps, warmup, sample, out, slot, barrier):
    m = MovingObjectRemoval(CFG, 4, 3, binding=orc)
    buf = np.empty((maxp, 8), np.float32)
    step = 0
    for phase, count in (("warm", warmup), ("timed", steps)):
        if phase == "timed" and barrier is not None:
            barrier.wait()
        t0 = time.perf_counter()
        for _ in range(count):
            f = step % sample
            if f == 0 and step:
                m = MovingObjectRemoval(CFG, 4, 3, binding=orc)  # replay: fresh tracker
            m.push_raw_cloud_and_pose(*frames[f])
            m.filter_cloud(buf)
            step += 1
        if phase == "timed":
            out[slot] = time.perf_counter() - t0
    if barrier is not None:
        barrier.wait()


def bench_config(world, frames_in_pool=None, frame_bytes=None):
    """The `config` object of the JSON line: identical for the GPU arm and the CPU arm (same workload, same parameters)."""
    return {"workload": WORKLOAD, "sequences_per_gpu": 1, "parallelism": f"replicas x{world} (independent sequences, no collective)",
            "l2": "no input is ever re-read: every step reads a frame no earlier step has read (K+W distinct frames staged in HBM / pinned host memory); "
                  "intermediates (~10 MB per frame) are L2-resident by design",
            "n_bad": 4, "n_good": 3, "mor_config": "config/MOR_config_hdl64.txt"}


def run_reference(args, rank, world):
    """CPU arm. The reference (ROS + PCL 1.8 + FLANN + Eigen) cannot be built offline, so this times the oracle port
    (kind "port"). The workload is ONE sensor sequence, as on the GPU arm, and the reference is strictly
    single-threaded per sequence (no threads / OpenMP anywhere in src/): `value` is therefore one thread on one
    sequence. The all-cores aggregate (one independent sequence per host thread - the C5-style workload) is
    reported beside it in `all_cores`, to be compared with the GPU arm's `multi_sequence` / `c5` figures."""
    if rank != 0:
        return
    orc = MorBinding(C.CDLL(str(ROOT / "oracle" / "libmor_oracle.so")), "oracle_")
    K, W = args.steps, args.warmup
    sample = 48  # bounded sample: the first 48 frames of the C2 sequence, replayed
    s = Synth(SCENARIO, 2)
    frames = [s.frame(f) for f in range(sample)]
    # K timed steps after W untimed ones, in both figures; the oracle needs ~0.1-0.3 s per frame on this sample
    t_single = [0.0]
    _oracle_worker(orc, frames, s.max_points, K, W, sample, t_single, 0, None)
    value = K / t_single[0]
    threads = max(1, min(os.cpu_count() or 1, 64))
    t_all = [0.0] * threads
    barrier = threading.Barrier(threads + 1)
    ths = [threading.Thread(target=_oracle_worker, args=(orc, frames, s.max_points, K, W, sample, t_all, t, barrier)) for t in range(threads)]
    for t in ths:
        t.start()
    barrier.wait()
    t0 = time.perf_counter()
    barrier.wait()
    dt = time.perf_counter() - t0
    for t in ths:
        t.join()
    all_cores = threads * K / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": 1e3 * t_single[0] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(world),
        "reference_arm": {"timed_steps": K, "note": "one sequence, one thread: the reference path is single-threaded per sensor stream"},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": 1, "kind": "port",
                         "sample": f"{K} frames replaying the first {sample} frames of C2, CPU oracle (PCL-semantics restatement, g++ -O2)",
                         "host_cpus": os.cpu_count()},
        "all_cores": {"value": all_cores, "unit": "frames/s", "cores": threads,
                      "sample": f"{threads} independent sequences (one per host thread), {K} frames each from the same {sample}-frame sample"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_cores(local_rank, world):
    """Each rank keeps to its own share of the host cores (rank r -> cores [r*c/w, (r+1)*c/w)): eight processes that
    share one host otherwise migrate over all cores and NUMA nodes while they feed their GPUs."""
    if world <= 1 or not hasattr(os, "sched_setaffinity"):
        return None
    try:
        cpus = sorted(os.sched_getaffinity(0))
        per = max(1, len(cpus) // world)
        mine = cpus[local_rank * per:(local_rank + 1) * per] or cpus
        os.sched_setaffinity(0, mine)
        return [mine[0], mine[-1]]
    except OSError:
        return None


def run_product(args, rank, local_rank, world):
    import torch  # device plumbing + torch.distributed only
    import torch.distributed as dist

    cores = bind_to_gpu_cores(local_rank, world)
    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    b = load_product()  # raises if the CUDA library is missing: no fallback
    K, W = args.steps, args.warmup
    F = K + W
    probe = Synth(SCENARIO, 2)
    maxp = probe.max_points
    pts, _pp = pinned_array(b, (F, maxp, 4), np.float32)
    out_host, _po = pinned_array(b, (maxp, 8), np.float32)
    npts = np.zeros(F, np.int64)
    poses = np.zeros((F, 7), np.float64)
    generate_frames(2 + rank, F, pts, npts, poses)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(local_rank)

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ------------------------------------------------------------------ e2e: host C ABI, pinned buffers
    m = MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp)
    for f in range(W):
        m.push_raw_cloud_and_pose(pts[f, : npts[f]], poses[f])
        m.filter_cloud(out_host)
    lat = np.zeros(K)
    d2h = 0
    # the timed loop calls the C ABI itself (what a C/C++ caller would do); pointers and pose arrays are prepared
    # outside so that the Python glue does not sit on the per-frame critical path
    in_ptrs = [C.c_void_p(pts[f].ctypes.data) for f in range(F)]
    pose_arrs = [(C.c_double * 7)(*poses[f]) for f in range(F)]
    ns = [int(v) for v in npts]
    out_ptr = C.c_void_p(out_host.ctypes.data)
    n_out = C.c_uint32(0)
    n_out_ref = C.byref(n_out)
    push_fn, filter_fn, hh = b.push, b.filter, m.h
    barrier()
    m.event_record(0)
    for i in range(K):
        f = W + i
        t0 = time.perf_counter()
        st1 = push_fn(hh, in_ptrs[f], ns[f], 16, 0, 4, 8, 12, pose_arrs[f])
        st2 = filter_fn(hh, out_ptr, maxp, n_out_ref)
        lat[i] = time.perf_counter() - t0
        if st1 or st2:
            raise RuntimeError(f"C ABI status {st1}/{st2} at frame {f}")
        d2h += n_out.value * 32 + 96
    m.event_record(1)
    e2e_ms = m.event_elapsed_ms(0, 1)
    barrier()
    e2e_ms = max_over_ranks(e2e_ms)
    crc_e2e_last = zlib.crc32(out_host[: n_out.value].tobytes())
    m.close()

    # ------------------------------------------------------------------ e2e, pipelined: mor_submit_frame / mor_collect_frame. Same frames, same
    # pinned buffers, every frame's H2D and D2H inside the timed region; the copies of frames f+1 and f-1 run beside the kernel of frame f
    # (results are delivered one call later). Wall clock from the first submit to the last collect.
    DEPTH = 4  # MOR_STREAM_DEPTH: frames in flight (results arrive DEPTH - 1 calls late)
    out_bufs = [out_host] + [pinned_array(b, (maxp, 8), np.float32)[0] for _ in range(DEPTH - 1)]
    out_ptrs = [C.c_void_p(o.ctypes.data) for o in out_bufs]
    m = MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp)
    m.set_pipelining(True)
    submit_fn, collect_fn, hh = b.submit_frame, b.collect_frame, m.h
    for f in range(W):
        if submit_fn(hh, in_ptrs[f], ns[f], 16, 0, 4, 8, 12, pose_arrs[f], out_ptrs[f % DEPTH], maxp) or collect_fn(hh, n_out_ref):
            raise RuntimeError("C ABI error in the streaming warm-up")
    barrier()
    d2h_s = 0
    t0 = time.perf_counter()
    for i in range(K):
        f = W + i
        st1 = submit_fn(hh, in_ptrs[f], ns[f], 16, 0, 4, 8, 12, pose_arrs[f], out_ptrs[f % DEPTH], maxp)
        st2 = collect_fn(hh, n_out_ref) if i >= DEPTH - 1 else 0
        if st1 or st2:
            raise RuntimeError(f"C ABI status {st1}/{st2} at streamed frame {f}")
        if i >= DEPTH - 1:
            d2h_s += n_out.value * 32 + 96
    for _ in range(min(DEPTH - 1, K)):
        if collect_fn(hh, n_out_ref):
            raise RuntimeError("C ABI error at the last streamed frames")
        d2h_s += n_out.value * 32 + 96
    stream_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    stream_ms = max_over_ranks(stream_ms)
    crc_stream_last = zlib.crc32(out_bufs[(F - 1) % DEPTH][: n_out.value].tobytes())
    m.close()

    # ------------------------------------------------------------------ device-resident: value
    d_frames = C.c_void_p()
    frame_bytes = maxp * 16
    assert b.device_alloc(local_rank, F * frame_bytes, C.byref(d_frames)) == 0
    assert b.device_upload(local_rank, d_frames, pts.ctypes.data_as(C.c_void_p), F * frame_bytes) == 0
    def device_resident(pipelining):
        """K frames through the device-resident calls, nothing asked back per frame. pipelining: mor_set_pipelining - the back half
        of frame f (transform, match, moving test, chain, filter) in ONE launch with the front half of frame f+1 (ingest ...
        cluster statistics) on disjoint SMs; the region ends when the last frame's back half has completed."""
        mm = MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp)
        mm.set_pipelining(pipelining)
        for f in range(W):
            mm.push_device(d_frames.value + f * frame_bytes, int(npts[f]), poses[f])
            mm.filter_device(None, 0, want_count=False)
        mm.sync()
        barrier()
        l0 = mm.launch_count()
        mm.event_record(0)
        for i in range(K):
            f = W + i
            mm.push_device(d_frames.value + f * frame_bytes, int(npts[f]), poses[f])
            mm.filter_device(None, 0, want_count=False)  # the filtered cloud stays in the handle's device buffer
        mm.sync()  # (pipelining: launches the back half of the last frame; the region covers K whole frames either way)
        mm.event_record(1)
        ms = mm.event_elapsed_ms(0, 1)
        barrier()
        n_launches = mm.launch_count() - l0
        ms = max_over_ranks(ms)
        cl = mm.counts()
        if cl["ERRFLAGS"]:
            raise RuntimeError(f"device capacity flags {cl['ERRFLAGS']}")
        # the timed run did the work: its last output equals the last output of the (independent) end-to-end run, byte for byte
        last = np.empty((cl["NOUT"], 8), np.float32)
        if last.size:
            assert b.device_download(local_rank, last.ctypes.data_as(C.c_void_p), C.c_void_p(mm.output_device()), last.nbytes) == 0
        crc_last = zlib.crc32(last.tobytes())
        mm.close()
        return ms, n_launches, crc_last, last

    one_ms, one_launches, crc_one_last, _ = device_resident(False)        # one kernel per frame: k_frame
    dev_ms, launches, crc_dev_last, dev_last = device_resident(True)      # the headline: k_frame_pipe
    launches_all = sum_over_ranks(launches)

    # ------------------------------------------------------------------ multi-sequence (C5-style): S independent sequences per GPU
    from dynamicslamtool_b200 import SequenceBatch
    multi = None
    S = args.sequences
    if S > 1:
        hs = [MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp) for _ in range(S)]
        d_outs = []
        for _ in range(S):
            p = C.c_void_p()
            assert b.device_alloc(local_rank, maxp * 32, C.byref(p)) == 0
            d_outs.append(p)
        offs = [(si * F) // S for si in range(S)]  # every sequence starts at its own frame of the pool and wraps around once
        batch = SequenceBatch(hs)
        outs = [p.value for p in d_outs]

        def steps(t0, t1):
            for t in range(t0, t1):
                fs = [(offs[si] + t) % F for si in range(S)]
                batch.step_device([d_frames.value + f * frame_bytes for f in fs], [int(npts[f]) for f in fs], [poses[f] for f in fs], outs)

        Wm = max(3, W)
        steps(0, Wm)
        hs[0].sync()
        barrier()
        l0m = hs[0].launch_count()
        hs[0].event_record(0)
        steps(Wm, Wm + K)
        hs[0].event_record(1)
        multi_ms = hs[0].event_elapsed_ms(0, 1)
        barrier()
        multi_ms = max_over_ranks(multi_ms)
        multi_launches = hs[0].launch_count() - l0m
        alg = 0.0
        for hh2 in hs:
            hh2.sync()
            alg += algorithmic_bytes(hh2.counts())
        peak_m, which_m = measured_peak_gbs()
        step_us = 1e3 * multi_ms / K
        multi = {"sequences_per_gpu": S, "value": world * S * K / (multi_ms * 1e-3), "unit": "frames/s", "ms_per_round": multi_ms / K,
                 "launches": multi_launches,
                 "roofline": {"bound": "hbm", "kernel": "k_frame_batch", "achieved": alg / (step_us * 1e-6) / 1e9, "peak": peak_m, "unit": "GB/s",
                              "frac": alg / (step_us * 1e-6) / 1e9 / peak_m, "peak_source": which_m, "algorithmic_bytes_per_launch": alg,
                              "kernel_avg_us": step_us, "note": "one launch per step: the step time is the kernel's duration (CUDA events on its stream)"},
                 "note": "device-resident, mor_batch_step_device: S sequences per launch of the frame kernel (a group of CTAs per sequence); aggregate over all sequences and GPUs"}
        for hh2 in hs:
            hh2.close()
        for p in d_outs:
            b.device_free(local_rank, p)

    # ------------------------------------------------------------------ C5: 128 sequences per GPU (1024 on 8 GPUs), 32 frames each, seeds 1000 + s
    c5 = None
    if args.c5_sequences > 0:
        c5 = run_c5(b, local_rank, rank, world, args.c5_sequences, 32, args.sequences if args.sequences > 1 else 37, maxp, max_over_ranks, sum_over_ranks, barrier)

    # ------------------------------------------------------------------ multi-sequence, end to end: one host thread per sequence through
    # the host C ABI (pinned input, H2D, kernels, D2H): copies of one sequence overlap the kernels of the others
    multi_e2e = None
    Se = min(args.e2e_sequences, 16)
    if Se > 1:
        hs2 = [MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp) for _ in range(Se)]
        outs2 = [pinned_array(b, (maxp, 8), np.float32) for _ in range(Se)]
        offs2 = [(si * F) // Se for si in range(Se)]
        gate = threading.Barrier(Se + 1)

        def drive(si):
            hh3, outp = hs2[si].h, C.c_void_p(outs2[si][0].ctypes.data)
            no = C.c_uint32(0)
            for phase, cnt in (("warm", 5), ("timed", K)):
                if phase == "timed":
                    gate.wait()
                for t in range(cnt):
                    f = (offs2[si] + (t if phase == "warm" else 5 + t)) % F
                    if b.push(hh3, in_ptrs[f], ns[f], 16, 0, 4, 8, 12, pose_arrs[f]) or b.filter(hh3, outp, maxp, C.byref(no)):
                        raise RuntimeError("C ABI error in the multi-sequence e2e leg")
            gate.wait()

        ths = [threading.Thread(target=drive, args=(si,)) for si in range(Se)]
        for th in ths:
            th.start()
        gate.wait()
        t0 = time.perf_counter()
        gate.wait()
        dt = time.perf_counter() - t0
        for th in ths:
            th.join()
        dt = max_over_ranks(dt)
        multi_e2e = {"sequences_per_gpu": Se, "value": world * Se * K / dt, "unit": "frames/s",
                     "note": "host C ABI, one host thread + stream per sequence, pinned buffers, H2D and D2H inside; wall clock over all sequences"}
        for hh3 in hs2:
            hh3.close()

    clocks = sampler.stop() if rank == 0 else None

    # ------------------------------------------------------------------ the frame kernel's duration and its phases (rank 0; outside the timed regions)
    roofline = None
    phases = {}
    frame_bytes_alg = 0.0
    if rank == 0:
        peak, which = measured_peak_gbs()
        # both passes time frames W .. F - 1, the K frames of the timed legs
        # pass 1: the fused kernel, one pair of CUDA events around every launch
        m2 = MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp)
        m2.set_timing(True)
        kern_ms, alg_sum, nc_sum, nprof = 0.0, 0, 0, 0
        timeline = {}
        for f in range(F):
            m2.push_device(d_frames.value + f * frame_bytes, int(npts[f]), poses[f])
            m2.filter_device(None, 0, want_count=True)
            if f >= W:
                kern_ms += m2.last_device_ms()[0]
                for k, v in m2.phase_times().items():
                    timeline[k] = timeline.get(k, 0.0) + v
                c = m2.counts()
                alg_sum += algorithmic_bytes(c)
                nc_sum += c["NC"]
                nprof += 1
        m2.close()
        nprof = max(nprof, 1)
        frame_bytes_alg = alg_sum / nprof
        kern_us = 1e3 * kern_ms / nprof
        traffic, traffic_note, traffic_pipe = None, None, None
        tp = ROOT / "profiles" / "traffic.json"
        if tp.exists():
            tj = json.loads(tp.read_text())
            traffic, traffic_note = tj.get("k_frame"), tj.get("note")
            traffic_pipe = tj.get("k_frame_pipe")
        pipe_us = 1e3 * dev_ms / K
        roofline = {"bound": "hbm", "kernel": "k_frame_pipe", "achieved": frame_bytes_alg / (pipe_us * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": frame_bytes_alg / (pipe_us * 1e-6) / 1e9 / peak, "traffic": traffic_pipe, "traffic_note": traffic_note, "peak_source": which,
                    "algorithmic_bytes_per_launch": frame_bytes_alg, "units_per_launch": 1, "bytes_per_unit": frame_bytes_alg,
                    "unit_note": "one launch = the back half of frame f + the front half of frame f+1 = one frame's worth of work; SURVEY 8(d): 16N + 17Nt + 104Nc + "
                                 "24Nk' + 32(P1+P2) + 20Nt + 16Nout from the frames' device-side counts",
                    "kernel_avg_us": pipe_us, "kernel_share_of_frame": 1.0,
                    "how": "the timed region is K back-to-back launches of this kernel on one stream (one launch per step): its average duration is the step time, CUDA events",
                    "mean_cloud_points": nc_sum / nprof,
                    "single_frame_kernel": {"kernel": "k_frame", "what": "the whole frame as ONE launch (the latency path: synchronous calls, no pipelining)",
                                            "kernel_avg_us": kern_us, "achieved": frame_bytes_alg / (kern_us * 1e-6) / 1e9,
                                            "frac": frame_bytes_alg / (kern_us * 1e-6) / 1e9 / peak, "traffic": traffic}}
        # pass 2: one launch per phase (the same device functions), each between events
        m2 = MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp)
        for f in range(W):
            m2.push_device(d_frames.value + f * frame_bytes, int(npts[f]), poses[f])
            m2.filter_device(None, 0, want_count=True)
        m2.set_kernel_profiling(True)
        for f in range(W, F):
            m2.push_device(d_frames.value + f * frame_bytes, int(npts[f]), poses[f])
            m2.filter_device(None, 0, want_count=True)
        prof = m2.kernel_profile()
        m2.set_kernel_profiling(False)
        m2.close()
        tot = sum(v[0] for v in prof.values()) or 1.0
        phases = {k: {"avg_us": 1e3 * v[0] / v[1], "launches": v[1], "share": v[0] / tot, "in_frame_kernel_us": timeline.get(k, 0.0) / nprof}
                  for k, v in prof.items() if v[1]}
        if "ph_link" in phases:
            mean_nc = nc_sum / nprof
            phases["ph_link"]["roofline"] = {"bytes_per_unit": 20, "units": mean_nc, "achieved_gbs": 20 * mean_nc / (phases["ph_link"]["avg_us"] * 1e-6) / 1e9,
                                             "frac": 20 * mean_nc / (phases["ph_link"]["avg_us"] * 1e-6) / 1e9 / peak}

    # ------------------------------------------------------------------ CPU baseline + parity spot check (rank 0, N = 1 only)
    cpu, spot = None, None
    if rank == 0 and world == 1 and not args.no_cpu:
        orc = MorBinding(C.CDLL(str(ROOT / "oracle" / "libmor_oracle.so")), "oracle_")
        mo = MovingObjectRemoval(CFG, 4, 3, binding=orc)
        out_o = np.empty((maxp, 8), np.float32)
        t_used = 0.0
        crcs_o = []
        for f in range(F):
            t0 = time.perf_counter()
            mo.push_raw_cloud_and_pose(pts[f, : npts[f]], poses[f])
            oo = mo.filter_cloud(out_o)
            if f >= W:
                t_used += time.perf_counter() - t0
            crcs_o.append((zlib.crc32(oo.tobytes()), zlib.crc32(mo.tap("removed_mask").tobytes())))
        cpu = {"value": K / t_used, "unit": "frames/s", "cores": 1, "kind": "port",
               "sample": f"frames {W}..{F - 1} of the same C2 sequence ({K} timed steps after {W} untimed), single thread, CPU oracle (PCL-semantics restatement, -O2)",
               "host_cpus": os.cpu_count()}
        # the same frames through the product, untimed: output cloud and removal mask of every frame against the oracle's
        mg = MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp)
        equal = 0
        first_bad = None
        for f in range(F):
            mg.push_raw_cloud_and_pose(pts[f, : npts[f]], poses[f])
            og = mg.filter_cloud(out_host)
            ok = (zlib.crc32(og.tobytes()), zlib.crc32(mg.tap("removed_mask").tobytes())) == crcs_o[f]
            equal += 1 if ok else 0
            if not ok and first_bad is None:
                first_bad = f
        spot = {"frames": F, "crc_equal": equal == F, "frames_equal": equal, "first_mismatch": first_bad,
                "what": "crc32 of the filtered cloud bytes and of the removed-point mask, product vs oracle, frame by frame from the start of the timed sequence",
                "timed_run_last_frame_crc_equal": crc_dev_last == crc_e2e_last,
                "timed_run_note": "last output of the device-resident timed run == last output of the end-to-end timed run (two independent full passes)",
                "timed_run_last_frame_equals_oracle": crcs_o[-1][0] == crc_dev_last}
        mg.close()
        # north_star: "any tie-breaking divergence at the exact clustering radius counted and reported": point pairs within
        # 2 ulps of r^2 (the pairs a differently rounded distance or a pruned kd-tree search could classify the other way),
        # counted by brute force on both sides for a few frames of the sequence
        mt = MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp)
        mo2 = MovingObjectRemoval(CFG, 4, 3, binding=orc)
        tie_frames, ties_gpu, ties_orc, pairs_checked = 0, 0, 0, 0
        for f in range(min(3, F)):
            mt.push_raw_cloud_and_pose(pts[f, : npts[f]], poses[f]); mt.filter_cloud(out_host)
            mo2.push_raw_cloud_and_pose(pts[f, : npts[f]], poses[f]); mo2.filter_cloud(out_o)
            ties_gpu += mt.radius_ties(2); ties_orc += mo2.radius_ties(2)
            nc_f = mt.counts()["NC"]
            pairs_checked += nc_f * (nc_f - 1) // 2
            tie_frames += 1
        spot["radius_ties"] = {"frames": tie_frames, "ulps": 2, "pairs_within_band": ties_gpu, "oracle_pairs_within_band": ties_orc,
                               "point_pairs_examined": pairs_checked,
                               "note": "pairs of cloud points with |d2 - r2| <= 2 ulp(r2): the only pairs on which a real PCL/FLANN build could cluster differently "
                                       "from the bit-exact strict `<` both sides evaluate; 0 means no such pair exists in these frames"}
        mt.close()

    # ------------------------------------------------------------------ the drop-in C++ class (what a user of the reference calls), rank 0, N = 1
    e2e_class = None
    harness = ROOT / "harness" / "mov_harness"
    if rank == 0 and world == 1 and harness.exists():
        import re
        import subprocess
        try:
            # the harness leaves its first 5 callbacks out of its summary: 5 + K frames = K timed callbacks
            r = subprocess.run([str(harness), str(CFG), "2", "2", str(5 + K), "--quiet"], capture_output=True, text=True, timeout=300,
                               env=dict(os.environ, CUDA_VISIBLE_DEVICES=str(local_rank)))
            m1 = re.search(r"summary frames (\d+) mean_ms ([\d.]+) p50_ms ([\d.]+) p99_ms ([\d.]+) fps ([\d.]+)", r.stdout)
            m2 = re.search(r"stages copy_ms ([\d.]+) push_ms ([\d.]+) filter_ms ([\d.]+)", r.stdout)
            if m1:
                e2e_class = {"frames": int(m1.group(1)), "ms_per_callback": float(m1.group(2)), "p50_ms": float(m1.group(3)), "p99_ms": float(m1.group(4)),
                             "value": float(m1.group(5)), "unit": "frames/s",
                             "stages_ms": {"copy_of_the_message": float(m2.group(1)), "pushRawCloudAndPose": float(m2.group(2)), "filterCloud": float(m2.group(3))} if m2 else None,
                             "how": "harness/mov_harness (the ROS-free external_sync_test.cpp): the C++ class MovingObjectRemoval, pageable PCLPointCloud2 input as a ROS "
                                    "callback has it, pushRawCloudAndPose + filterCloud + `output` filled per frame, host wall clock per callback"}
        except Exception as ex:  # the class-level figure is a side measurement: never fail the bench line over it
            e2e_class = {"error": str(ex)}

    b.device_free(local_rank, d_frames)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    value = world * K / (dev_ms * 1e-3)
    e2e_value = world * K / (e2e_ms * 1e-3)
    peak, which = measured_peak_gbs()
    cfg = bench_config(world)
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dev_ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "value_how": "device-resident calls with mor_set_pipelining: one k_frame_pipe launch per step = back half of frame f beside the front half of frame f+1 on disjoint "
                     "SM groups; K whole frames inside the timed region (the last back half included); `unpipelined` = one k_frame launch per frame",
        "config": cfg,
        "clocks": clocks,
        "e2e": {"value": world * K / (stream_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": int(np.mean(npts[W:]) * 16 + 56), "d2h_bytes_per_step": int(d2h_s / K),
                "ms_per_step": stream_ms / K,
                "how": "host C ABI, pinned host buffers, mor_submit_frame + mor_collect_frame: every frame's H2D, frame kernel and D2H inside the timed region (wall clock, "
                       "first submit to last collect, max over ranks); up to four frames in flight, pipelined launches (mor_set_pipelining): copies of neighbouring frames overlap the kernels, results arrive three calls later",
                "last_frame_crc_equals_serial": crc_stream_last == crc_e2e_last,
                "serial": {"value": e2e_value, "unit": "frames/s", "ms_per_step": e2e_ms / K, "d2h_bytes_per_step": int(d2h / K),
                           "how": "mor_push_raw_cloud_and_pose + mor_filter_cloud per frame, nothing overlapped (the reference's callback protocol): per-frame latency",
                           "latency_ms": {"p50": float(np.percentile(lat, 50) * 1e3), "p99": float(np.percentile(lat, 99) * 1e3), "max": float(lat.max() * 1e3)}}},
        "gpu_launches": int(launches_all),
        "unpipelined": {"value": world * K / (one_ms * 1e-3), "unit": "frames/s", "ms_per_step": one_ms / K, "launches": int(one_launches),
                        "what": "the same K frames with one k_frame launch per frame (no overlap of consecutive frames): the per-frame device latency",
                        "last_frame_crc_equals_pipelined": crc_one_last == crc_dev_last},
        "roofline": roofline,
        "frame_roofline": {"algorithmic_bytes_per_frame": frame_bytes_alg, "achieved_gbs": frame_bytes_alg * (K / (dev_ms * 1e-3)) / 1e9,
                           "frac": frame_bytes_alg * (K / (dev_ms * 1e-3)) / 1e9 / peak, "peak": peak, "peak_source": which},
        "phases": phases,
        "multi_sequence": multi,
        "c5": c5,
        "multi_sequence_e2e": multi_e2e,
        "e2e_class": e2e_class,
        "cpu_baseline": cpu,
        "parity_spot_check": spot,
        "host": {"staged_frames": F, "staged_mb": F * frame_bytes / 1e6, "rank_cores": cores},
    }
    if args.dump_outputs:
        # what a caller of the headline path receives for its last timed frame (frame W + K - 1 of seed 2): the filtered
        # cloud, float32 [n_out, 8] PointXYZI wire records (x, y, z, 1, intensity, 0, 0, 0); at most 133,312 x 32 B
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        np.save(out_dir / "filtered_cloud.npy", dev_last)
    print(json.dumps(line), flush=True)


def run_c5(b, local_rank, rank, world, per_gpu, T, S, maxp, max_over_ranks, sum_over_ranks, barrier):
    """BASELINE config 5 as SURVEY 8(d) words it: independent C2-shaped sequences with seeds 1000 + s, 32 frames each,
    sequence s -> rank s mod world; `per_gpu` sequences per GPU (128 => the full 1024 on 8 GPUs: weak scaling). The
    sequences of a rank are taken S at a time: generated on the host and staged in HBM (untimed: the generator is not
    the subject), handles reset, then T batched steps timed with CUDA events on the launching stream."""
    from concurrent.futures import ThreadPoolExecutor
    from dynamicslamtool_b200 import SequenceBatch
    total = per_gpu * world
    mine = [s for s in range(total) if s % world == rank]
    frame_bytes = maxp * 16
    d_in = C.c_void_p()
    assert b.device_alloc(local_rank, S * T * frame_bytes, C.byref(d_in)) == 0
    d_outs = []
    for _ in range(S):
        p = C.c_void_p()
        assert b.device_alloc(local_rank, maxp * 32, C.byref(p)) == 0
        d_outs.append(p)
    hs = [MovingObjectRemoval(CFG, 4, 3, device=local_rank, binding=b, max_points=maxp) for _ in range(S)]
    threads = max(1, (os.cpu_count() or 8) // max(1, min(world, 8)))

    def generate(seq):
        syn = Synth(SCENARIO, 1000 + seq)
        syn.threads = 1  # the pool below already runs one sequence per host thread
        return [syn.frame(f) for f in range(T)]

    timed_ms, frames_done, launches, gen_s, out_pts = 0.0, 0, 0, 0.0, 0
    batch_ms = []
    for b0 in range(0, len(mine), S):
        seqs = mine[b0:b0 + S]
        t0 = time.time()
        with ThreadPoolExecutor(threads) as ex:
            data = list(ex.map(generate, seqs))
        gen_s += time.time() - t0
        for si, frames in enumerate(data):
            for f, (p, _) in enumerate(frames):
                assert b.device_upload(local_rank, C.c_void_p(d_in.value + (si * T + f) * frame_bytes), p.ctypes.data_as(C.c_void_p), p.nbytes) == 0
        group = hs[:len(seqs)]
        batch = SequenceBatch(group)
        lead = group[0]

        def step(f):
            batch.step_device([d_in.value + (si * T + f) * frame_bytes for si in range(len(seqs))], [int(data[si][f][0].shape[0]) for si in range(len(seqs))],
                              [data[si][f][1] for si in range(len(seqs))], [p.value for p in d_outs[:len(seqs)]])

        # untimed warm-up (the GPU has idled through seconds of host-side generation and upload: its clocks are down), then
        # the handles go back to "no frame seen" and the batch's T frames are timed from frame 0
        for h in group:
            h.reset()
        for f in range(min(3, T)):
            step(f)
        lead.sync()
        for h in group:
            h.reset()
        l0 = lead.launch_count()
        lead.event_record(0)
        for f in range(T):
            step(f)
        lead.event_record(1)
        lead.sync()
        batch_ms.append(lead.event_elapsed_ms(0, 1))
        timed_ms += batch_ms[-1]
        launches += lead.launch_count() - l0
        frames_done += len(seqs) * T
        for h in group:
            h.sync()
            c = h.counts()
            if c["ERRFLAGS"]:
                raise RuntimeError(f"C5: device capacity flags {c['ERRFLAGS']}")
            out_pts += c["NOUT"]
    for h in hs:
        h.close()
    for p in d_outs:
        b.device_free(local_rank, p)
    b.device_free(local_rank, d_in)
    barrier()
    worst = max_over_ranks(timed_ms)
    frames_all = sum_over_ranks(frames_done)
    return {"workload": f"C5: {total} independent C2-shaped sequences (seeds 1000..{1000 + total - 1}), {T} frames each, sequence s -> rank s mod {world}, "
                        f"{S} sequences per launch", "sequences": total, "sequences_per_gpu": per_gpu, "frames": int(frames_all),
            "value": frames_all / (worst * 1e-3), "unit": "frames/s", "timed_ms_max_over_ranks": worst, "launches_rank0": launches,
            "generator_seconds_rank0": gen_s, "batch_ms_rank0": [round(v, 2) for v in batch_ms], "output_points_last_frames_rank0": out_pts, "data": "synthetic, staged in HBM before the timed region"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps (frames per sequence) of every leg on the C2 workload; the C5 leg keeps its 32 frames per sequence")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--e2e-sequences", type=int, default=8, help="sequences (= host threads) of the multi-sequence end-to-end figure (1 = skip)")
    ap.add_argument("--sequences", type=int, default=37, help="independent sequences per launch for the multi_sequence figure and the batches of the C5 leg (37 = a group of 4 CTAs per sequence on 148 SMs; 1 = skip)")
    ap.add_argument("--c5-sequences", type=int, default=128, help="BASELINE config 5: sequences per GPU (128 x 8 GPUs = the full 1024), 32 frames each (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the headline path's output of its last step as DIR/filtered_cloud.npy "
                                                          "(rank 0; the inputs depend on --steps and --warmup only)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_product(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
