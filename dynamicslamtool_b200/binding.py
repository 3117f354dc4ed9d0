"""ctypes binding of the mor_b200 C ABI (include/mor_b200.h).

`MorBinding(lib, prefix)` wraps any shared library that exports the ABI under a symbol prefix:
the product library `libmor_b200.so` (prefix ``mor_``, CUDA, sm_100a) and - from tests/bench only -
the CPU oracle (prefix ``oracle_``). The product loader never falls back to anything: if the CUDA
library is missing it raises.

Reference surface mirrored here (prabinrath/dynamicslamtool):
  MovingObjectRemoval(nh, config_path, n_bad, n_good)   include/MOR/MovingObjectRemoval.h:160
  pushRawCloudAndPose(cloud, pose)                      include/MOR/MovingObjectRemoval.h:163
  filterCloud(cloud, f_id) / output                     include/MOR/MovingObjectRemoval.h:159,166
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
REPO_ROOT = PKG_DIR.parent
PRODUCT_LIB = Path(os.environ["MOR_PRODUCT_LIB"]) if os.environ.get("MOR_PRODUCT_LIB") else PKG_DIR / "libmor_b200.so"  # (debug builds)
SYNTH_LIB = PKG_DIR / "libmor_synth.so"

NO_FIELD = 0xFFFFFFFF

STATUS = {
    0: "MOR_OK", 1: "MOR_ERR_CONFIG_OPEN", 2: "MOR_ERR_CONFIG_KEY", 3: "MOR_ERR_CONFIG_VALUE",
    4: "MOR_ERR_CONFIG_MISSING", 5: "MOR_ERR_ARG", 6: "MOR_ERR_CAPACITY", 7: "MOR_ERR_CUDA", 8: "MOR_ERR_STATE",
}

# tap ids (mor_tap_id) -> (name, numpy dtype, trailing shape)
TAPS = {
    "counts": (0, np.int32, ()),
    "point_class": (1, np.uint8, ()),
    "labels": (2, np.int32, ()),
    "cluster_id": (3, np.int32, ()),
    "cluster_root": (4, np.int32, ()),
    "cluster_size": (5, np.int32, ()),
    "centroids": (6, np.float32, (3,)),
    "transform": (7, np.float32, ()),
    "prev_centroids_t": (8, np.float32, (3,)),
    "prev_points_t": (9, np.float32, (3,)),
    "match_query": (10, np.int32, ()),
    "match_match": (11, np.int32, ()),
    "match_dist": (12, np.float32, ()),
    "match_score": (13, np.float64, ()),
    "flags": (14, np.uint8, ()),
    "mo_centroids": (15, np.float32, (3,)),
    "mo_conf": (16, np.int32, ()),
    "removed_mask": (17, np.uint8, ()),
    "cluster_removed": (18, np.uint8, ()),
    "recip_query": (19, np.int32, ()),
    "recip_match": (20, np.int32, ()),
    "ground_voxels": (21, np.float32, (8,)),
    "cluster_bbox": (22, np.float32, (6,)),
    "prev_bbox_t": (23, np.float32, (6,)),
}

COUNT_NAMES = ["N", "NT", "NC", "NG", "K", "KPREV", "M", "NMO", "NOUT", "NKPREV", "P1", "P2", "TWO_FRAMES",
               "EXTRACT_OVERFLOW", "MU", "NCPREV", "NK", "NVOX", "FRAME", "ERRFLAGS", "SIZE_TIES"]


class MorConfig(C.Structure):
    _fields_ = (
        [(n, C.c_float) for n in ("gp_limit", "gp_leaf", "bin_gap", "volume_constraint", "pde_lb", "pde_ub",
                                  "leave_off_distance", "catch_up_distance", "trim_x", "trim_y", "trim_z",
                                  "ec_distance_threshold", "pde_distance_threshold")]
        + [("min_cluster_size", C.c_int64), ("max_cluster_size", C.c_int64)]
        + [("method_choice", C.c_int32), ("opc_normalization_factor", C.c_int32), ("ground_mode", C.c_int32)]
        + [("gp_planarity", C.c_float), ("gp_bin_width", C.c_float), ("n_bad", C.c_int32), ("n_good", C.c_int32)]
        + [(n, C.c_char * 64) for n in ("output_topic", "debug_topic", "marker_topic", "input_pointcloud_topic",
                                        "input_odometry_topic", "output_fid", "debug_fid")]
    )


class MorLimits(C.Structure):
    _fields_ = [("max_points", C.c_uint32), ("max_clusters", C.c_uint32), ("max_moving", C.c_uint32), ("max_cells", C.c_uint32),
                ("reserved", C.c_uint32 * 4)]


class MorBatchFrame(C.Structure):
    _fields_ = [("d_data", C.c_void_p), ("n", C.c_uint32), ("point_step", C.c_uint32), ("off_x", C.c_uint32), ("off_y", C.c_uint32),
                ("off_z", C.c_uint32), ("off_i", C.c_uint32), ("pose7", C.c_double * 7), ("d_out", C.c_void_p)]


MARKER_DTYPE = np.dtype([("position", np.float32, 3), ("scale", np.float32, 3), ("color", np.float32, 4), ("id", np.int32), ("cluster", np.int32)])


class MorError(RuntimeError):
    def __init__(self, status: int, where: str, detail: str = ""):
        self.status = status
        super().__init__(f"{where}: {STATUS.get(status, status)} {detail}".strip())


class MorBinding:
    """Function table of one library exporting the ABI under `prefix`."""

    def __init__(self, lib: C.CDLL, prefix: str):
        self.lib, self.prefix = lib, prefix
        f = self._fn
        vp, u32, sz = C.c_void_p, C.c_uint32, C.c_size_t
        self.create_ex = f("create_ex", [C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(MorLimits), C.POINTER(vp)])
        self.destroy = f("destroy", [vp])
        self.reset = f("reset", [vp])
        self.get_config = f("get_config", [vp, C.POINTER(MorConfig)])
        self.parse_config = f("parse_config", [C.c_char_p, C.POINTER(MorConfig)])
        self.push = f("push_raw_cloud_and_pose", [vp, vp, u32, u32, u32, u32, u32, u32, C.POINTER(C.c_double)])
        self.filter = f("filter_cloud", [vp, vp, u32, C.POINTER(u32)])
        self.sync = f("sync", [vp])
        self.tap = f("tap", [vp, C.c_int, vp, sz, C.POINTER(sz)])
        self.get_cluster_collection = f("get_cluster_collection", [vp, vp, u32, C.POINTER(u32)])
        self.get_moving_markers = f("get_moving_markers", [vp, vp, u32, C.POINTER(u32)])
        self.count_radius_ties = f("count_radius_ties", [vp, C.c_int, C.POINTER(C.c_uint64)])
        # product-only entry points (absent from the oracle)
        self.get_limits = f("get_limits", [vp, C.POINTER(MorLimits)], True)
        self.push_device = f("push_raw_cloud_and_pose_device", [vp, vp, u32, u32, u32, u32, u32, u32, C.POINTER(C.c_double)], True)
        self.filter_device = f("filter_cloud_device", [vp, vp, u32, C.POINTER(u32)], True)
        self.get_output_device = f("get_output_device", [vp, C.POINTER(vp)], True)
        self.alloc_pinned = f("alloc_pinned", [sz, C.POINTER(vp)], True)
        self.free_pinned = f("free_pinned", [vp], True)
        self.device_alloc = f("device_alloc", [C.c_int, sz, C.POINTER(vp)], True)
        self.device_free = f("device_free", [C.c_int, vp], True)
        self.device_upload = f("device_upload", [C.c_int, vp, vp, sz], True)
        self.device_download = f("device_download", [C.c_int, vp, vp, sz], True)
        self.get_launch_count = f("get_launch_count", [vp, C.POINTER(C.c_uint64)], True)
        self.get_last_device_ms = f("get_last_device_ms", [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)], True)
        self.set_timing = f("set_timing", [vp, C.c_int], True)
        self.last_error = f("last_error", [vp], True, C.c_char_p)
        self.batch_step_device = f("batch_step_device", [C.POINTER(vp), u32, C.POINTER(vp), C.POINTER(u32), u32, u32, u32, u32, u32,
                                                         C.POINTER(C.c_double), C.POINTER(vp)], True)
        self.batch_step_device_mixed = f("batch_step_device_mixed", [C.POINTER(vp), u32, C.POINTER(MorBatchFrame)], True)
        self.event_record = f("event_record", [vp, C.c_int], True)
        self.event_elapsed_ms = f("event_elapsed_ms", [vp, C.c_int, C.c_int, C.POINTER(C.c_float)], True)
        self.set_kernel_profiling = f("set_kernel_profiling", [vp, C.c_int], True)
        self.get_kernel_profile = f("get_kernel_profile", [vp, C.c_int, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64)], True)
        self.get_phase_times = f("get_phase_times", [vp, C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_int)], True)
        self.phase_name = f("phase_name", [C.c_int], True, C.c_char_p)
        self.submit_frame = f("submit_frame", [vp, vp, u32, u32, u32, u32, u32, u32, C.POINTER(C.c_double), vp, u32], True)
        self.collect_frame = f("collect_frame", [vp, C.POINTER(u32)], True)
        self.frames_in_flight = f("frames_in_flight", [vp, C.POINTER(u32)], True)
        self.set_pipelining = f("set_pipelining", [vp, C.c_int], True)
        self.set_output_records = f("set_output_records", [vp, C.c_int], True)

    def _fn(self, name, argtypes, optional=False, restype=C.c_int):
        try:
            fn = getattr(self.lib, self.prefix + name)
        except AttributeError:
            if optional:
                return None
            raise
        fn.argtypes, fn.restype = argtypes, restype
        return fn


_product = None


def load_product() -> MorBinding:
    """Load the CUDA product library. Fails loudly - there is no CPU fallback."""
    global _product
    if _product is None:
        if not PRODUCT_LIB.exists():
            raise RuntimeError(f"{PRODUCT_LIB} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(nvcc, sm_100a). There is no CPU fallback for the MOR hot path.")
        _product = MorBinding(C.CDLL(str(PRODUCT_LIB)), "mor_")
    return _product


def parse_config(path, binding: MorBinding | None = None) -> MorConfig:
    b = binding or load_product()
    cfg = MorConfig()
    st = b.parse_config(str(path).encode(), C.byref(cfg))
    if st:
        raise MorError(st, "parse_config", str(path))
    return cfg


class MovingObjectRemoval:
    """Python mirror of the reference class (include/MOR/MovingObjectRemoval.h:96-168) over the C ABI.

    push_raw_cloud_and_pose(points, pose7): `points` is a C-contiguous numpy array; either float32
    [N, F] with x,y,z,intensity in columns 0..3 (F >= 3; F == 3 => no intensity), or a uint8 blob with
    explicit point_step/offsets (PCLPointCloud2 semantics, reference cpp:523).
    filter_cloud() returns float32 [N_out, 8] PointXYZI wire records (x,y,z,1,intensity,0,0,0), cpp:690; with
    set_output_records(True), uint8 [N_out, point_step] copies of the input records the points came from.
    """

    def __init__(self, config_path, n_bad: int = 4, n_good: int = 3, device: int = 0, binding: MorBinding | None = None,
                 max_points: int = 0, max_clusters: int = 0, max_moving: int = 0, max_cells: int = 0):
        self.b = binding or load_product()
        self.h = C.c_void_p()
        lim = MorLimits(max_points=max_points, max_clusters=max_clusters, max_moving=max_moving, max_cells=max_cells)
        st = self.b.create_ex(str(config_path).encode(), n_bad, n_good, device, C.byref(lim), C.byref(self.h))
        if st:
            self.h = C.c_void_p()
            raise MorError(st, "mor_create", str(config_path))
        self._out = None
        self.n_input = 0
        self.output_records = False  # the setting (set_output_records)
        self._rec_step = 0           # point_step of the last frame pushed in record mode, 0 for PointXYZI output

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.b.destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st, where):
        if st:
            detail = ""
            if self.b.last_error is not None:
                e = self.b.last_error(self.h)
                detail = e.decode() if e else ""
            raise MorError(st, where, detail)

    @property
    def config(self) -> MorConfig:
        cfg = MorConfig()
        self._check(self.b.get_config(self.h, C.byref(cfg)), "get_config")
        return cfg

    def reset(self):
        """Forget every frame seen so far (a freshly constructed object with the same configuration)."""
        self._check(self.b.reset(self.h), "reset")

    @property
    def limits(self) -> MorLimits:
        lim = MorLimits()
        self._check(self.b.get_limits(self.h, C.byref(lim)), "get_limits")
        return lim

    def push_raw_cloud_and_pose(self, points: np.ndarray, pose7, point_step=None, offsets=None):
        pose = (C.c_double * 7)(*[float(v) for v in pose7])
        if points.dtype == np.float32 and point_step is None:
            assert points.ndim == 2 and points.shape[1] >= 3 and points.flags.c_contiguous
            n, step = points.shape[0], points.shape[1] * 4
            offs = (0, 4, 8, 12 if points.shape[1] >= 4 else NO_FIELD)
        else:
            assert points.flags.c_contiguous and point_step is not None and offsets is not None
            n, step, offs = points.nbytes // point_step, point_step, offsets
        self._keep = points  # the copy is asynchronous: keep the buffer alive until the next sync
        self.n_input = n
        self._check(self.b.push(self.h, points.ctypes.data_as(C.c_void_p), n, step, *offs, pose), "push_raw_cloud_and_pose")
        self._rec_step = step if self.output_records else 0

    def _out_array(self, cap, step):
        """Default output buffer: float32 [cap, 8] PointXYZI records, or uint8 [cap, step] input records."""
        if self._out is None or self._out.shape[0] < cap or self._out.dtype != (np.uint8 if step else np.float32) \
                or (step and self._out.shape[1] != step):
            self._out = np.empty((cap, step), np.uint8) if step else np.empty((cap, 8), np.float32)
        return self._out

    def filter_cloud(self, out: np.ndarray | None = None) -> np.ndarray:
        cap = max(self.n_input, 1)
        if out is None:
            out = self._out_array(cap, self._rec_step)
        n_out = C.c_uint32(0)
        self._check(self.b.filter(self.h, out.ctypes.data_as(C.c_void_p), out.shape[0], C.byref(n_out)), "filter_cloud")
        return out[: n_out.value]

    def set_output_records(self, enabled: bool):
        """Deliver the filtered cloud as copies of the input records (every field kept) from the next push on; see
        mor_set_output_records. filter_cloud / collect_frame then return uint8 [N_out, point_step] arrays."""
        self._check(self.b.set_output_records(self.h, 1 if enabled else 0), "set_output_records")
        self.output_records = bool(enabled)

    def cluster_collection(self) -> np.ndarray:
        """The reference's VISUALIZE debug cloud (cpp:226-229, :553-558): float32 [N_k, 8] PointXYZI records."""
        n = C.c_uint32(0)
        self._check(self.b.get_cluster_collection(self.h, None, 0, C.byref(n)), "get_cluster_collection")
        out = np.empty((n.value, 8), np.float32)
        if n.value:
            self._check(self.b.get_cluster_collection(self.h, out.ctypes.data_as(C.c_void_p), n.value, C.byref(n)), "get_cluster_collection")
        return out

    def moving_markers(self) -> np.ndarray:
        """Bounding-box markers of the last filter_cloud (cpp:640-642), structured array of MARKER_DTYPE."""
        n = C.c_uint32(0)
        self._check(self.b.get_moving_markers(self.h, None, 0, C.byref(n)), "get_moving_markers")
        out = np.zeros(n.value, MARKER_DTYPE)
        if n.value:
            self._check(self.b.get_moving_markers(self.h, out.ctypes.data_as(C.c_void_p), n.value, C.byref(n)), "get_moving_markers")
        return out

    def radius_ties(self, ulps: int = 2) -> int:
        """Point pairs of the current cloud within `ulps` units in the last place of the squared clustering radius."""
        v = C.c_uint64(0)
        self._check(self.b.count_radius_ties(self.h, ulps, C.byref(v)), "count_radius_ties")
        return v.value

    def sync(self):
        self._check(self.b.sync(self.h), "sync")

    def tap(self, name: str) -> np.ndarray:
        tid, dt, trail = TAPS[name]
        nb = C.c_size_t(0)
        st = self.b.tap(self.h, tid, None, 0, C.byref(nb))
        if st not in (0, 6):
            self._check(st, f"tap({name})")
        buf = np.empty(nb.value, np.uint8)
        if nb.value:
            self._check(self.b.tap(self.h, tid, buf.ctypes.data_as(C.c_void_p), nb.value, C.byref(nb)), f"tap({name})")
        arr = buf.view(dt)
        return arr.reshape((-1,) + trail) if trail else arr

    def counts(self) -> dict:
        c = self.tap("counts")
        return {n: int(c[i]) for i, n in enumerate(COUNT_NAMES)}

    # device-resident variants (product only)
    def push_device(self, d_ptr: int, n: int, pose7, point_step=16, offsets=(0, 4, 8, 12)):
        pose = (C.c_double * 7)(*[float(v) for v in pose7])
        self.n_input = n
        self._check(self.b.push_device(self.h, C.c_void_p(d_ptr), n, point_step, *offsets, pose), "push_device")

    def filter_device(self, d_out: int | None, cap: int, want_count=True) -> int:
        """d_out None: the records stay in the handle's own device buffer (output_device())."""
        n_out = C.c_uint32(0)
        self._check(self.b.filter_device(self.h, C.c_void_p(d_out) if d_out else None, cap, C.byref(n_out) if want_count else None), "filter_device")
        return n_out.value

    def output_device(self) -> int:
        p = C.c_void_p()
        self._check(self.b.get_output_device(self.h, C.byref(p)), "get_output_device")
        return p.value

    # pipelined streaming (product only): copies of neighbouring frames overlap the frame kernel
    def submit_frame(self, points: np.ndarray, pose7, out: np.ndarray, point_step=None, offsets=None):
        """push + filter of one frame, enqueued without waiting; `points` and `out` (float32 [cap, 8], or uint8
        [cap, point_step] with output records; both ideally views of pinned memory) must stay untouched until
        collect_frame() has returned for this frame."""
        pose = (C.c_double * 7)(*[float(v) for v in pose7])
        if points.dtype == np.float32 and point_step is None:
            assert points.ndim == 2 and points.shape[1] >= 3 and points.flags.c_contiguous
            n, step = points.shape[0], points.shape[1] * 4
            offs = (0, 4, 8, 12 if points.shape[1] >= 4 else NO_FIELD)
        else:
            assert points.flags.c_contiguous and point_step is not None and offsets is not None
            n, step, offs = points.nbytes // point_step, point_step, offsets
        if self.output_records:
            assert out.dtype == np.uint8 and out.ndim == 2 and out.shape[1] == step and out.flags.c_contiguous
        else:
            assert out.dtype == np.float32 and out.ndim == 2 and out.shape[1] == 8 and out.flags.c_contiguous
        self.n_input = n
        self._inflight = getattr(self, "_inflight", [])
        self._inflight.append((points, out))
        st = self.b.submit_frame(self.h, points.ctypes.data_as(C.c_void_p), n, step, *offs, pose, out.ctypes.data_as(C.c_void_p), out.shape[0])
        if st:
            self._inflight.pop()
        self._check(st, "submit_frame")

    def collect_frame(self) -> np.ndarray:
        """Waits for the oldest submitted frame; returns the filled part of the `out` it was submitted with."""
        n_out = C.c_uint32(0)
        st = self.b.collect_frame(self.h, C.byref(n_out))
        q = getattr(self, "_inflight", [])
        out = q.pop(0)[1] if q else None
        self._check(st, "collect_frame")
        return out[: n_out.value]

    def set_pipelining(self, enabled: bool):
        """Throughput mode: the back half of a frame runs beside the front half of the next one (see mor_set_pipelining)."""
        self._check(self.b.set_pipelining(self.h, 1 if enabled else 0), "set_pipelining")

    def frames_in_flight(self) -> int:
        v = C.c_uint32(0)
        self._check(self.b.frames_in_flight(self.h, C.byref(v)), "frames_in_flight")
        return v.value

    def event_record(self, slot: int):
        self._check(self.b.event_record(self.h, slot), "event_record")

    def event_elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_float(0)
        self._check(self.b.event_elapsed_ms(self.h, a, b, C.byref(ms)), "event_elapsed_ms")
        return ms.value

    def set_kernel_profiling(self, enabled: bool):
        self._check(self.b.set_kernel_profiling(self.h, 1 if enabled else 0), "set_kernel_profiling")

    def kernel_profile(self) -> dict:
        """{kernel name: (total_ms, launches)} accumulated since profiling was enabled."""
        out, i = {}, 0
        while True:
            name = C.create_string_buffer(32)
            ms, n = C.c_double(0), C.c_uint64(0)
            if self.b.get_kernel_profile(self.h, i, name, C.byref(ms), C.byref(n)):
                break
            out[name.value.decode()] = (ms.value, n.value)
            i += 1
        return out

    def phase_times(self) -> dict:
        """{phase name: microseconds} of the last frame kernel (its own %globaltimer timeline, barriers included)."""
        us = (C.c_float * 32)()
        n = C.c_int(0)
        self._check(self.b.get_phase_times(self.h, us, 32, C.byref(n)), "get_phase_times")
        return {self.b.phase_name(i).decode(): float(us[i]) for i in range(n.value)}

    def set_timing(self, enabled: bool):
        self._check(self.b.set_timing(self.h, 1 if enabled else 0), "set_timing")

    def last_device_ms(self):
        a, b = C.c_float(0), C.c_float(0)
        self._check(self.b.get_last_device_ms(self.h, C.byref(a), C.byref(b)), "get_last_device_ms")
        return a.value, b.value

    def launch_count(self) -> int:
        v = C.c_uint64(0)
        self._check(self.b.get_launch_count(self.h, C.byref(v)), "get_launch_count")
        return v.value


class SequenceBatch:
    """S independent sequences stepped with one set of kernel launches (mor_batch_step_device, BASELINE config 5)."""

    def __init__(self, handles: list[MovingObjectRemoval]):
        self.handles = handles
        self.b = handles[0].b
        S = len(handles)
        self._hs = (C.c_void_p * S)(*[h.h.value for h in handles])
        self._data = (C.c_void_p * S)()
        self._out = (C.c_void_p * S)()
        self._n = (C.c_uint32 * S)()
        self._poses = (C.c_double * (7 * S))()

    def step_device(self, d_ptrs, ns, poses, d_outs, point_step=16, offsets=(0, 4, 8, 12)):
        """d_outs[s] must hold ns[s] output points: 32-byte PointXYZI records, or ns[s] * point_step bytes when the
        handles deliver output records (set_output_records)."""
        S = len(self.handles)
        for s in range(S):
            self._data[s] = d_ptrs[s]
            self._out[s] = d_outs[s]
            self._n[s] = int(ns[s])
            self.handles[s].n_input = int(ns[s])
            for k in range(7):
                self._poses[7 * s + k] = float(poses[s][k])
        st = self.b.batch_step_device(self._hs, S, self._data, self._n, point_step, *offsets, self._poses, self._out)
        if st:
            self.handles[0]._check(st, "batch_step_device")


class MixedBatch:
    """One step of S sequences that may differ in frame count, configuration, limits, record layout and output records
    (mor_batch_step_device_mixed). The handles may change from one step to the next."""

    def __init__(self, binding: MorBinding | None = None):
        self.b = binding or load_product()

    def step(self, handles: list[MovingObjectRemoval], d_ptrs, ns, poses, d_outs, point_steps=None, offsets=None):
        """Per sequence s: device records d_ptrs[s] (ns[s] of point_steps[s] bytes, default 16, field offsets offsets[s],
        default (0, 4, 8, 12)), pose poses[s]; d_outs[s] must hold ns[s] output records of the handle's output mode."""
        S = len(handles)
        hs = (C.c_void_p * S)(*[h.h.value for h in handles])
        frames = (MorBatchFrame * S)()
        for s in range(S):
            fr = frames[s]
            fr.d_data, fr.n, fr.d_out = d_ptrs[s], int(ns[s]), d_outs[s]
            fr.point_step = int(point_steps[s]) if point_steps is not None else 16
            fr.off_x, fr.off_y, fr.off_z, fr.off_i = offsets[s] if offsets is not None else (0, 4, 8, 12)
            for k in range(7):
                fr.pose7[k] = float(poses[s][k])
        st = self.b.batch_step_device_mixed(hs, S, frames)
        if st:
            handles[0]._check(st, "batch_step_device_mixed")
        for s in range(S):
            handles[s].n_input = int(ns[s])


class Synth:
    """Seeded synthetic LiDAR sequence (csrc/mor_synth.cpp). scenario 1..4 = C1..C4 of SURVEY §8d."""

    _lib = None

    def __init__(self, scenario: int, seed: int):
        if Synth._lib is None:
            if not SYNTH_LIB.exists():
                raise RuntimeError(f"{SYNTH_LIB} is missing: run __graft_entry__.build()")
            lib = C.CDLL(str(SYNTH_LIB))
            lib.mor_synth_create.argtypes = [C.c_int, C.c_uint64, C.POINTER(C.c_void_p)]
            lib.mor_synth_destroy.argtypes = [C.c_void_p]
            lib.mor_synth_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_double)]
            lib.mor_synth_frame.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32),
                                            C.POINTER(C.c_double), C.c_int]
            Synth._lib = lib
        self.h = C.c_void_p()
        if Synth._lib.mor_synth_create(scenario, seed, C.byref(self.h)):
            raise ValueError("bad scenario")
        mp, nf, hz = C.c_uint32(), C.c_uint32(), C.c_double()
        Synth._lib.mor_synth_info(self.h, C.byref(mp), C.byref(nf), C.byref(hz))
        self.max_points, self.nominal_frames, self.rate_hz = mp.value, nf.value, hz.value
        self.threads = min(os.cpu_count() or 1, 16)

    def frame(self, idx: int, out: np.ndarray | None = None):
        """Returns (points float32 [n,4], pose7 float64 [7])."""
        buf = out if out is not None else np.empty((self.max_points, 4), np.float32)
        n = C.c_uint32()
        pose = (C.c_double * 7)()
        st = Synth._lib.mor_synth_frame(self.h, idx, buf.ctypes.data_as(C.c_void_p), buf.shape[0], C.byref(n), pose, self.threads)
        if st:
            raise RuntimeError(f"mor_synth_frame -> {st}")
        pts = buf[: n.value]
        return (pts if out is not None else np.ascontiguousarray(pts)), np.array(pose[:], np.float64)

    def __del__(self):
        try:
            if self.h.value:
                Synth._lib.mor_synth_destroy(self.h)
        except Exception:
            pass
