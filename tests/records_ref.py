"""Input record layouts and the expected filtered cloud in record layout (mor_set_output_records), derived from the CPU
oracle's own bookkeeping: output point o is the input record of the o-th source index, where the sources are the kept
`cloud` points in ascending input order (point class 1, removal mask not 2), then the ground points in ascending input
order (point class 2) - ExtractIndices(negative) + the ground append of filterCloud, cpp:673-684."""
from __future__ import annotations

import numpy as np

from dynamicslamtool_b200.binding import NO_FIELD

PAD = 0xA5

# name -> (point_step, (off_x, off_y, off_z, off_i), extra fields {name: (offset, dtype)})
LAYOUTS = {
    "xyzi16": (16, (0, 4, 8, 12), {}),
    "xyzirt22": (22, (0, 4, 8, 12), {"ring": (16, "<u2"), "time": (18, "<f4")}),  # velodyne driver XYZIRT
    "odd13": (13, (1, 5, 9, NO_FIELD), {}),
    "odd19": (19, (3, 7, 11, 15), {}),
    "xyz12": (12, (0, 4, 8, NO_FIELD), {}),
}


def make_records(pts: np.ndarray, layout: str) -> tuple[np.ndarray, int, tuple]:
    """pts float32 [n, 4] -> (uint8 [n, point_step] records, point_step, offsets). Padding bytes are 0xA5; ring is the
    beam row (i % 16) and time a distinct float32 per point."""
    step, offs, extra = LAYOUTS[layout]
    n = len(pts)
    rec = np.full((n, step), PAD, np.uint8)
    for col, off in enumerate(offs):
        if off != NO_FIELD:
            rec[:, off:off + 4] = np.ascontiguousarray(pts[:, col]).view(np.uint8).reshape(n, 4)
    idx = np.arange(n)
    for name, (off, dt) in extra.items():
        v = (idx % 16).astype(dt) if name == "ring" else (idx.astype(np.float64) * 1e-6 + 0.25).astype(dt)
        size = np.dtype(dt).itemsize
        rec[:, off:off + size] = np.ascontiguousarray(v).view(np.uint8).reshape(n, size)
    return np.ascontiguousarray(rec), step, offs


def expected_sources(orc) -> np.ndarray:
    """Input index of every output point of the oracle's last filter_cloud."""
    pc, rm = orc.tap("point_class"), orc.tap("removed_mask")
    kept = np.flatnonzero((pc == 1) & (rm != 2))
    ground = np.flatnonzero(pc == 2)
    return np.concatenate([kept, ground])


def expected_records(orc, rec: np.ndarray) -> np.ndarray:
    return rec[expected_sources(orc)]


def fields_of(rec: np.ndarray, offs) -> np.ndarray:
    """float32 [n, 4] x, y, z, intensity (0 without an intensity field) read from records."""
    n = len(rec)
    out = np.zeros((n, 4), np.float32)
    for col, off in enumerate(offs):
        if off != NO_FIELD:
            out[:, col] = np.ascontiguousarray(rec[:, off:off + 4]).view(np.float32).reshape(n)
    return out
